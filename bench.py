#!/usr/bin/env python
"""bench.py - headline benchmark of the decoder-query + PDE-residual hot path on B200.

    python bench.py --gpus 1 --steps 20 --warmup 3                # our arm, 1 GPU
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N   # our arm, N GPUs (weak scaling)
    python bench.py --impl reference --steps K --warmup W          # the reference's CPU path (oracle port)
    python bench.py --steps 20 --warmup 3 --dump-outputs DIR       # also writes the last timed call's outputs as DIR/*.npy

Metric (BASELINE.json): PDE-residual query points/sec for forward + Jacobian + residual + backward on the
0.25 degree configuration (145x257 grid geometry, batch 8, 65 536 query points per sample).  A "step" is one
call of the fused operator on one batch of synthetic inputs.

  value  whole-job points/s with inputs resident in HBM: one dpn_pde_fwd_bwd call per step and rank (all its
         kernels), plus, for N > 1, the NCCL all-reduce of the decoder parameter gradients the call produced.
  e2e    the same metric through the reference-facing API, InterfacePhysics.place_one_batch(host tensors):
         pinned host -> device copies of every per-step input, PyTorch encoder + hyper-network, fused operator,
         backward through hyper-network and encoder, gradient all-reduce (N > 1), loss.item().
  roofline / cpu_baseline / clocks: see DESIGN.md section 7.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALGO_FLOP_PER_POINT = 31.89e6      # SURVEY.md 8(d): fwd + Jacobian + bwd, GEMM work only
# contraction FLOPs of the executed algorithm (DESIGN.md section 3): pass 1 + pass 2 + weight gradients, 6 nets, 2 FLOP per MAC;
# the split modes run pass 2 as the forward pass of the combined row WITHOUT its third GEMM (163 840 MACs: the column sum of gz comes
# out of the dWa contraction), the bf16 mode as the tangent chain (179 200)
EXEC_FLOP = {m: 6 * 2 * (407040 + p2 + 228352) for m, p2 in (('f16x3', 163840), ('f16x3a', 163840), ('bf16x3', 163840), ('bf16', 179200), ('fp32', 179200))}
MMA_PASSES = {"bf16": 1, "bf16x3": 3, "f16x3": 3, "f16x3a": 3, "fp32": 1}   # tensor-core MMAs issued per contraction (split operands: 3)
# ... except the two contractions whose A operand is the exact 0 / 1 ReLU mask (G4 of pass 1, dWa): 2 MMAs.  FLOPs as ISSUED to the pipe:
ISSUED_FLOP = {m: MMA_PASSES[m] * EXEC_FLOP[m] - (6 * 2 * 2 * 65536 if m in ("f16x3", "f16x3a", "bf16x3") else 0) for m in EXEC_FLOP}
DTYPE = {"bf16": "bf16", "bf16x3": "bf16 hi+lo (3 MMAs), fp32 accumulate", "f16x3": "fp16 hi+lo scaled (3 MMAs), fp32 accumulate",
         "f16x3a": "fp16 hi+lo scaled (3 MMAs, cross terms first), fp32 accumulate", "fp32": "f32"}
METRIC = "pde_residual_query_points_per_sec_fwd_jacobian_bwd"
UNIT = "points/s"

META_CFG = dict(name="TransformerNet", enc_in=2405, c_out=256, d_model=256, n_heads=8, e_layers=4, d_ff=256,
                dropout=0.5, activation="gelu", output_attention=False)
NET_CFG = dict(name="PhysicsNet", in_channels=192, hidden_channels=256, out_channels=1, token_num=159,
               learnable_token_num=256)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return dict(bf16=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))),
                    bf16_burst=float(d.get("bf16_tflops", 1590.0)), hbm=float(d.get("hbm_gbs", 6650.0)), source="measured")
    return dict(bf16=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def __enter__(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        return False

    def summary(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if not self.path or not os.path.exists(self.path):
            return out
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def _reference_step_factory(n_points, device):
    """One fwd+bwd step of the reference's path on `device` for B=1 x n_points query points.  Returns (step, kind, threads):
    kind "reference" = the UNMODIFIED reference - InterfacePhysics.place_one_batch (interface_physics.py:271-320) + backward(),
    imported from its tree through oracle/ref_harness.py (stubs for GDAL / xarray only; present in the build container, absent
    on a GPU box unless DPN_REFERENCE_ROOT points at a copy) - otherwise kind "port" = oracle/dpn_oracle.py (the restatement
    pinned to the reference's golden vectors) + this package's PyTorch encoder."""
    import torch
    from oracle import dpn_oracle as O
    from oracle import ref_harness as RH
    gen = torch.Generator().manual_seed(1234)
    x, y, t, f, cd = (a.to(device) for a in O.synthetic_points(n_points, gen))
    field = torch.randn(1, 159, 2405, generator=gen).to(device)
    if RH.available():
        m, builder_loss, cfg = RH.build_reference_model(seed=0)
        m = m.to(device)
        crit = builder_loss(name="MSELoss")
        lf = cfg["train_cfg"]["losses"]["loss_factor"]
        fh = torch.tensor([[[24.0 / 360.0]]], device=device)

        def step():
            m.physics_net.zero_grad(set_to_none=True)
            xs, ys, ts = (a.detach().clone().requires_grad_(True) for a in (x, y, t))
            loss = m.place_one_batch(xs, ys, ts, f, field, cd, fh, crit, lf, 0, 0, device, None, "inter")
            loss.backward()
            return loss
        return step, "reference", m
    from deepphysinet_b200.physics_net import PhysicsNet
    torch.manual_seed(0)
    net = PhysicsNet(META_CFG, NET_CFG).to(device)
    fh = torch.tensor([[[24.0 / 360.0]]], device=device)
    params = O.split_params(dict(net.named_parameters()))

    def step():
        net.zero_grad(set_to_none=True)
        meta = net.meta_net(field, fh)
        total, _ = O.place_one_batch(x, y, t, f, cd, fh, meta, params)
        total.backward()
        return total
    return step, "port", net


def cpu_reference_arm(steps, warmup, n_points, emit=True, as_baseline=False, n_gpus=1):
    """The reference's CPU path on all host threads, one sample of n_points query points per step, backward included
    (the unmodified reference when its tree is present, else the oracle port: _reference_step_factory)."""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    step, kind, _keep = _reference_step_factory(n_points, "cpu")
    what = ("unmodified reference InterfacePhysics.place_one_batch + backward" if kind == "reference"
            else "oracle port of place_one_batch + backward")

    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        float(step().detach())
        times.append(time.perf_counter() - t0)
    if as_baseline:
        best = min(times)
        return dict(value=n_points / best, unit=UNIT, cores=torch.get_num_threads(), kind=kind,
                    sample="B=1 x %d query points of the same workload, %s incl. encoder, best of %d after %d warm-up"
                           % (n_points, what, steps, warmup))
    mean = sum(times) / len(times)
    val = n_points / mean
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": "configs[1] 0.25deg grid (145x257), batch 8 x 65536 query points - bounded CPU sample per step",
                       "sample_points_per_step": n_points},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                             "sample": "B=1 x %d query points per step, %s incl. encoder" % (n_points, what)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if emit:
        _emit(line)
    return line


def eager_gpu_arm(dev, n_points):
    """The competitor on the same box (SURVEY 8(d)): the reference's formulation - six nets, one autograd.grad(create_graph=True)
    per derivative, double backward - executed by PyTorch eager on this GPU in fp32: the unmodified reference when its tree is
    present (kind "reference"), else the oracle port moved to CUDA (kind "port").  A baseline leg like cpu_baseline: reported
    beside the product, never part of it.  B = 1 x n_points, encoder included."""
    import torch
    try:
        step, kind, _keep = _reference_step_factory(n_points, dev)
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        out = {"value": n_points / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "kind": kind,
               "sample": "B=1 x %d query points, PyTorch eager fp32 autograd double backward (%s on cuda), incl. encoder" % (n_points, kind)}
        del step, _keep
    except Exception as ex:                                                  # a baseline leg must never take the bench down
        out = {"unavailable": str(ex)[:200]}
    torch.cuda.empty_cache()
    return out


_JSON_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line (the contract).  Libraries write there too - NCCL prints its version banner on
    stdout during the first collective whatever NCCL_DEBUG says - so file descriptor 1 is pointed at stderr for the whole run and
    the JSON line goes to a private duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, (json.dumps(line) + "\n").encode())


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(path, arrays):
    """Writes every array as path/<name>.npy, float64 where the call returns float64 and float32 otherwise, DUMP_BYTES at most
    in all.  Over that budget the smaller arrays are kept whole and each larger one is replaced by a sample of its flattened
    elements at sorted indices drawn from a fixed seed, so two runs with the same arguments store the same elements."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    budget = DUMP_BYTES - 1024 * len(arrays)                         # room for the .npy headers
    for i, (name, a) in enumerate(sorted(arrays.items(), key=lambda kv: (kv[1].nbytes, kv[0]))):
        share = budget // (len(arrays) - i)
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a)
        budget -= a.nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="f16x3", choices=["f16x3", "f16x3a", "bf16x3", "bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--points", type=int, default=65536)
    ap.add_argument("--cpu-points", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-modes", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2] / configs[3] legs (1 GPU only)")
    ap.add_argument("--no-eager-gpu", action="store_true", help="skip the PyTorch-eager-on-this-GPU baseline leg")
    ap.add_argument("--no-sustained", action="store_true", help="skip the 60-step power-capped steady-state timing of the same call")
    ap.add_argument("--no-graph", action="store_true", help="time the eager place_one_batch call instead of its CUDA-graph capture")
    ap.add_argument("--e2e-breakdown", action="store_true", help="print per-phase times of the e2e step to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed call returned on rank 0 (total loss, per-sample loss "
                         "terms, gradients of the 13 decoder weight tensors) as DIR/<name>.npy, %d MB at most" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    _claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            cpu_reference_arm(args.steps, args.warmup, args.cpu_points, n_gpus=args.gpus)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    ge.build()
    from deepphysinet_b200 import InterfacePhysics, functional as Fn, parallel as P, _native as Nat
    from deepphysinet_b200.config import DEFAULT_LOSS_FACTOR, DEFAULT_OBS_NORM

    rank, local_rank, world = P.init_from_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.backends.cudnn.allow_tf32 = False
    B, Np = args.batch, args.points

    obs = {k: dict(v, norm_type="mean_norm", use_norm=True) for k, v in DEFAULT_OBS_NORM.items()}
    torch.manual_seed(0)                                               # identical replicas on every rank
    model = InterfacePhysics(META_CFG, NET_CFG, obs, None, dict(img_size=(145, 257), dx=27000, dy=27000)).to(dev)
    model.mode = args.mode
    consts = model.consts(DEFAULT_LOSS_FACTOR)

    # synthetic inputs per SURVEY 8(d), per-rank seed (each rank owns B different samples: weak scaling)
    g = torch.Generator().manual_seed(100 + rank)
    hx = (torch.rand(B, Np, generator=g) * 256 * 27000.0).pin_memory()
    hy = torch.rand(B, Np, generator=g) * 144
    hf = (2 * 7.29e-5 * torch.sin((18.0 + hy * 0.25) / 180 * 3.141592653589793)).pin_memory()
    hy = (hy * 27000.0).pin_memory()
    ht = (torch.randint(0, 25, (B, Np), generator=g).float() * 3600.0).pin_memory()
    hcd = (0.5 * torch.randn(B, Np, 6, generator=g)).pin_memory()
    hfield = torch.randn(B, 159, 2405, generator=g).pin_memory()
    hfh = torch.full((B, 1, 1), 24.0 / 360.0).pin_memory()
    dx_, dy_, dt_, df_, dcd = (a.to(dev) for a in (hx, hy, ht, hf, hcd))
    with torch.no_grad():
        W = model.physics_net.decoder_weights(hfield.to(dev), hfh.to(dev))
    leaves = [w.detach().clone().requires_grad_(True) for w in W]
    static_idx = [5, 6, 7, 8, 9, 10, 11, 12]                           # Wd bd Wa ba Wb bb wo bo: parameter gradients
    n_static = sum(leaves[i].numel() for i in static_idx)
    flat = torch.zeros(n_static + 6, device=dev)

    holder = {}

    def op_step():
        total, terms = Fn.pde_residual(dx_, dy_, dt_, df_, dcd, Fn.DecoderWeights(*leaves), consts=consts, mode=args.mode)
        holder["launches"] = Nat.lib().dpn_last_launch_count()
        holder["last_total"], holder["last_terms"] = total, terms
        if world > 1:
            grads = total.grad_fn.grads if hasattr(total.grad_fn, "grads") else None
            off = 0
            if grads is not None:
                for i in static_idx:
                    n = grads[i].numel()
                    flat[off:off + n].copy_(grads[i].reshape(-1))
                    off += n
            flat[n_static:].copy_(terms.mean(0).float())
            dist.all_reduce(flat)
        return total

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return P.allreduce_max(e0.elapsed_time(e1) / steps, dev)

    if os.environ.get("DPN_DEBUG_FLAGS") or os.environ.get("DPN_PHASE_DEBUG") or os.environ.get("DPN_LIB_OVERRIDE"):
        raise SystemExit("bench.py measures the shipped library: unset DPN_DEBUG_FLAGS / DPN_PHASE_DEBUG / DPN_LIB_OVERRIDE")
    first_total = float(op_step().detach())                          # reference value of the loss for the checksum below
    with ClockSampler(local_rank) as clk:
        ms = timed(op_step, args.steps, args.warmup)
    clocks = clk.summary()
    pts_step = B * Np * world
    value = pts_step / (ms * 1e-3)
    # the timed op really computed the loss: finite, and identical (up to the order of the fp64 atomics) on every step
    last_total = float(holder["last_total"].detach())
    terms_mean = [float(v) for v in holder["last_terms"].mean(0).tolist()]
    if not (last_total == last_total and abs(last_total) < float("inf")) or abs(last_total - first_total) > 1e-6 * abs(first_total):
        raise SystemExit("timed operator returned loss %r, first call %r" % (last_total, first_total))
    checksum = {"total": last_total, "terms_mean_over_samples": terms_mean, "first_call_total": first_total}
    if args.dump_outputs and rank == 0:
        # the gradients are those backward() hands a caller of the last timed call (the call computed them already).  The inputs
        # are bit-identical from run to run, the outputs are not: the kernels accumulate with atomics, and two runs of the
        # default workload differed by up to 2.5e-7 of each gradient tensor's largest element (B200, 1000 W power limit)
        grads = torch.autograd.grad(holder["last_total"], leaves)
        outs = {"total": holder["last_total"], "terms": holder["last_terms"]}
        outs.update(("grad_" + n, g) for n, g in zip(Nat.WEIGHT_FIELDS, grads))
        dump_outputs(args.dump_outputs, {k: v.detach().cpu().numpy() for k, v in outs.items()})

    # ---- the same operator SUSTAINED: the B200 runs this call at its board power cap; after ~0.3 s of load the SM clock settles at
    # 1.4-1.5 GHz and a step takes ~8 % longer than in the first 20 steps after idle that `value` is timed over.  Reported beside it. ----
    sustained = None
    if not args.no_sustained:
        with ClockSampler(local_rank) as clk_s:
            ms_s = timed(op_step, 60, 30)
        sustained = {"value": pts_step / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s, "steps": 60, "warmup": 30,
                     "clocks": clk_s.summary(),
                     "note": "same call, timed after 30 further warm-up steps (power-capped steady state)"}

    # ---- strong scaling (SURVEY 8(d) C5: configs[1] sharded over the ranks), N > 1 only: total batch fixed at 8 samples ----
    strong = None
    if world > 1:
        s_steps = max(3, min(args.steps, 10))
        # level 1: samples sharded (8 / world per rank), all-reduce of the static-decoder gradients as in the weak-scaling op
        Bs = max(1, 8 // world)
        l1 = [w_[:Bs].detach().clone().requires_grad_(True) if i < 5 else leaves[i] for i, w_ in enumerate(leaves)]

        def strong_samples():
            total, terms = Fn.pde_residual(dx_[:Bs], dy_[:Bs], dt_[:Bs], df_[:Bs], dcd[:Bs], Fn.DecoderWeights(*l1), consts=consts, mode=args.mode)
            grads = total.grad_fn.grads
            off = 0
            for i in static_idx:
                n = grads[i].numel()
                flat[off:off + n].copy_(grads[i].reshape(-1))
                off += n
            flat[n_static:].copy_(terms.mean(0).float())
            dist.all_reduce(flat)
            return total
        ms_s1 = timed(strong_samples, s_steps, 3)
        # level 2: every rank holds all 8 samples and 1 / world of each sample's points (n_norm = all points); EVERY gradient the
        # call produces is a partial sum, generated weights included: one all-reduce (sum) of all 13 tensors
        lo, hi = P.shard_range(Np, rank, world)
        sl = lambda a: a[:, lo:hi].contiguous()
        px, py, pt_, pf, pcd = sl(dx_), sl(dy_), sl(dt_), sl(df_), sl(dcd)
        flat_all = torch.zeros(sum(w_.numel() for w_ in leaves) + 6 * B, device=dev)

        def strong_points():
            total, terms = Fn.pde_residual(px, py, pt_, pf, pcd, Fn.DecoderWeights(*leaves), consts=consts, mode=args.mode, n_norm=Np)
            grads = total.grad_fn.grads
            off = 0
            for g_ in grads:
                flat_all[off:off + g_.numel()].copy_(g_.reshape(-1))
                off += g_.numel()
            flat_all[off:].copy_(terms.reshape(-1).float())
            dist.all_reduce(flat_all)
            return total
        ms_s2 = timed(strong_points, s_steps, 3)
        tot_pts = 8 * Np if world <= 8 else Bs * world * Np
        strong = {"scaling": "strong", "batch_total": Bs * world, "points_per_sample": Np,
                  "samples_sharded": {"value": Bs * world * Np / (ms_s1 * 1e-3), "unit": UNIT, "ms_per_step": ms_s1, "samples_per_rank": Bs,
                                      "collective": "all-reduce of static-decoder gradients + loss terms (%.1f MB)" % (flat.numel() * 4 / 2 ** 20)},
                  "points_sharded": {"value": B * Np / (ms_s2 * 1e-3), "unit": UNIT, "ms_per_step": ms_s2, "points_per_rank_and_sample": hi - lo,
                                     "collective": "all-reduce (sum) of all 13 gradient tensors + loss terms (%.1f MB)" % (flat_all.numel() * 4 / 2 ** 20)},
                  "steps": s_steps}

    # ---- e2e through the reference-facing API, host buffers ----
    e2e = None
    if not args.no_e2e:
        reducer = P.FlatGradAllReduce(model.physics_net.parameters())
        crit = torch.nn.MSELoss()

        def e2e_step():
            model.physics_net.zero_grad(set_to_none=True)
            loss = model.place_one_batch(hx, hy, ht, hf, hfield, hcd, hfh, crit, DEFAULT_LOSS_FACTOR, 0, rank, dev)
            loss.backward()
            reducer()
            return loss.item()

        if args.e2e_breakdown:
            def phase_times():
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
                t0 = time.perf_counter()
                model.physics_net.zero_grad(set_to_none=True)
                ev[0].record()
                dev_in = [a.to(dev, non_blocking=True) for a in (hx, hy, ht, hf, hfield, hcd, hfh)]
                ev[1].record()
                Wd_ = model.physics_net.decoder_weights(dev_in[4], dev_in[6])
                ev[2].record()
                tot, _ = Fn.pde_residual(dev_in[0], dev_in[1], dev_in[2], dev_in[3], dev_in[5], Wd_, consts=consts, mode=args.mode)
                ev[3].record()
                tot.backward()
                ev[4].record()
                reducer()
                ev[5].record()
                t1 = time.perf_counter()
                tot.item()
                t2 = time.perf_counter()
                names = ["h2d", "encoder+hypernet fwd", "fused op", "backward (hypernet+encoder)", "grad all-reduce"]
                return {n: ev[i].elapsed_time(ev[i + 1]) for i, n in enumerate(names)} | {"cpu_issue_ms": (t1 - t0) * 1e3, "wall_ms": (t2 - t0) * 1e3}
            for _ in range(3):
                phase_times()
            print("[rank %d] e2e phases (ms): %s" % (rank, json.dumps(phase_times())), file=sys.stderr)
        e_steps = max(3, min(args.steps, 10))
        api = "InterfacePhysics.place_one_batch(host tensors) + backward + grad all-reduce + loss.item()"
        step_fn = e2e_step
        if not args.no_graph:
            # the same call captured once into a CUDA graph (deepphysinet_b200.graphed): pinned-host -> device copies, encoder,
            # fused operator and backward replay as ONE launch; the NCCL all-reduce and loss.item() stay outside the graph
            try:
                from deepphysinet_b200.graphed import PrefetchedPlaceOneBatch
                gstep = PrefetchedPlaceOneBatch(model, (hx, hy, ht, hf, hfield, hcd, hfh), crit, DEFAULT_LOSS_FACTOR, dev, rank=rank)
                gstep.prefetch()                                               # the first batch; every step below issues the next one

                def graphed_step():
                    loss = gstep()                                             # graph replay on the batch prefetched last
                    gstep.prefetch()                                           # this step's H2D (all inputs, pinned host -> device): runs
                    reducer()                                                  # on the copy stream underneath the compute just enqueued
                    return loss.item()
                ref_loss = e2e_step()
                got_loss = graphed_step()
                if abs(got_loss - ref_loss) > 1e-3 * abs(ref_loss):
                    raise RuntimeError("graphed step loss %r != eager loss %r" % (got_loss, ref_loss))
                step_fn = graphed_step
                api = ("PrefetchedPlaceOneBatch (CUDA graph of place_one_batch + backward; the step's pinned-host -> device copies "
                       "double-buffered on a copy stream) + grad all-reduce + loss.item()")
            except Exception as ex:                                            # host-side orchestration only: report and time the eager call
                print("[rank %d] CUDA-graph capture of the e2e step failed (%s): timing the eager call" % (rank, ex), file=sys.stderr)
        ms_e = timed(step_fn, e_steps, max(5, args.warmup))
        h2d = sum(a.numel() * a.element_size() for a in (hx, hy, ht, hf, hcd, hfield, hfh))
        e2e = {"value": pts_step / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * world,
               "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e, "steps_per_s": 1e3 / ms_e, "steps": e_steps, "api": api}
        if not args.no_sustained:                                               # same call in the power-capped steady state (see `sustained`)
            ms_es = timed(step_fn, 40, 20)
            e2e["sustained_ms_per_step"] = ms_es
            e2e["sustained_value"] = pts_step / (ms_es * 1e-3)
        if step_fn is not e2e_step:
            ms_eager = timed(e2e_step, e_steps, 3)
            e2e["eager_ms_per_step"] = ms_eager

    # ---- the other arithmetic modes, for the record (fewer steps; accuracy of each in DESIGN.md section 6) ----
    modes = {}
    if rank == 0 and world == 1 and not args.no_modes:
        notes = {"f16x3": "tcgen05, scaled fp16 hi+lo operands: fp32-class accuracy (2e-6..8e-6 vs fp64 oracle)",
                 "f16x3a": "f16x3 with cross-first accumulation of the mask-deciding GEMMs: pre-activation error 2.6x smaller (values 7e-8)",
                 "bf16x3": "tcgen05, bf16 hi+lo operands: 1e-4..4e-3 vs fp64 oracle",
                 "bf16": "tcgen05, plain bf16 operands: 2e-2..9e-2 on Jacobian / gradients",
                 "fp32": "CUDA-core fp32 FMA, the reference arithmetic: 5e-7 vs fp64 oracle"}
        for m in ("f16x3", "f16x3a", "bf16x3", "bf16", "fp32"):
            if m == args.mode:
                continue
            def m_step(m=m):
                return Fn.pde_residual(dx_, dy_, dt_, df_, dcd, Fn.DecoderWeights(*leaves), consts=consts, mode=m)[0]
            n_m = 3 if m == "fp32" else 8
            for _ in range(3):
                m_step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n_m):
                m_step()
            e1.record()
            torch.cuda.synchronize()
            ms_m = e0.elapsed_time(e1) / n_m
            modes[m] = {"value": B * Np / (ms_m * 1e-3), "unit": UNIT, "ms_per_step": ms_m, "note": notes[m]}
            if m == "fp32":                                  # CUDA-core mode: executed FLOPs against the MEASURED FP32 FFMA peak (tools/ffma_peak.cu)
                try:
                    ffma = json.load(open(os.path.join(ROOT, "profiles", "ffma_peak.json")))["fp32_ffma_tflops_sustained"]
                    ex = EXEC_FLOP[m] * modes[m]["value"] / 1e12
                    modes[m]["roofline"] = {"bound": "fp32 FFMA", "achieved": ex, "peak": ffma, "unit": "TFLOP/s", "frac": ex / ffma,
                                            "note": "executed contraction FLOPs (%.2f MFLOP/point)" % (EXEC_FLOP[m] / 1e6)}
                except Exception:
                    pass

    # ---- the other single-GPU configurations of BASELINE.json, a few steps each ----
    configs = {}
    if rank == 0 and world == 1 and not args.no_configs:
        def time_it(fn, n):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        # configs[2]: fused decoder + Jacobian + residual + backward microbench, one sample, 1M - 16M random query points
        micro = {}
        l1 = [w_[:1].detach().clone().requires_grad_(True) if i < 5 else leaves[i] for i, w_ in enumerate(leaves)]
        for logn in (20, 22, 24):
            n_ = 1 << logn
            gq = torch.Generator(device=dev).manual_seed(logn)
            qx = torch.rand(1, n_, generator=gq, device=dev) * 256 * 27000.0
            qy = torch.rand(1, n_, generator=gq, device=dev) * 144
            qf = 2 * 7.29e-5 * torch.sin((18.0 + qy * 0.25) / 180 * 3.141592653589793)
            qy = qy * 27000.0
            qt = torch.randint(0, 25, (1, n_), generator=gq, device=dev).float() * 3600.0
            qcd = 0.5 * torch.randn(1, n_, 6, generator=gq, device=dev)
            ms_c = time_it(lambda: Fn.pde_residual(qx, qy, qt, qf, qcd, Fn.DecoderWeights(*l1), consts=consts, mode=args.mode), 2)
            micro["2^%d" % logn] = {"value": n_ / (ms_c * 1e-3), "unit": UNIT, "ms_per_step": ms_c}
            del qx, qy, qf, qt, qcd
        configs["configs[2] microbench B=1, fwd+Jacobian+residual+bwd"] = micro
        # configs[3]: continuous-time dense-grid inference, 145 x 257 nodes x 48 hourly leads, values only (no residuals)
        coarse = torch.randn(1, 5, 37, 65, 6, device=dev)
        fd, fh1 = hfield[:1].to(dev), hfh[:1].to(dev)
        leads = list(range(48))
        model.pred_t_span = 48 * 3600.0                                       # one window spanning the 48 leads
        ms_g = time_it(lambda: model.predict_grid(fd, coarse, fh1, leads), 3)
        with torch.no_grad():
            Wg = model.physics_net.decoder_weights(fd, fh1)
        ms_gc = time_it(lambda: model.predict_grid(fd, coarse, fh1, leads, weights=Wg), 3)
        model.pred_t_span = 86400
        npts = 145 * 257 * 48
        configs["configs[3] dense-grid inference 145x257 x 48 leads, values only"] = {
            "value": npts / (ms_g * 1e-3), "unit": "grid points/s", "ms_per_sweep": ms_g, "points": npts,
            "with_cached_generated_weights": {"value": npts / (ms_gc * 1e-3), "ms_per_sweep": ms_gc}}
        del coarse
        torch.cuda.empty_cache()

    pk = peaks()
    per_gpu_pts = B * Np / (ms * 1e-3)
    achieved = ALGO_FLOP_PER_POINT * per_gpu_pts / 1e12
    roof_file = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    traffic = None
    if os.path.exists(roof_file):
        try:
            traffic = json.load(open(roof_file)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "tensor", "achieved": achieved, "peak": pk["bf16"], "unit": "TFLOP/s", "frac": achieved / pk["bf16"],
                "traffic": traffic,
                "kernel": "dpn_pde_fwd_bwd: all kernels of one call (pass1_ts / pass2z / wgrad2 tcgen05 kernels + encode, residual, scale plan)",
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (%s)" % pk["source"],
                "algorithmic_flop_per_point": ALGO_FLOP_PER_POINT, "executed_flop_per_point": EXEC_FLOP[args.mode],
                "executed_tflops": EXEC_FLOP[args.mode] * per_gpu_pts / 1e12,
                "mma_passes_per_contraction": MMA_PASSES[args.mode],
                "tensor_pipe_tflops": ISSUED_FLOP[args.mode] * per_gpu_pts / 1e12}

    # ---- the reference's own way of running this path on the same GPU: PyTorch eager autograd (double backward) ----
    eager_gpu = None
    if rank == 0 and world == 1 and not args.no_eager_gpu:
        eager_gpu = eager_gpu_arm(dev, args.points)

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_reference_arm(3, 1, args.cpu_points, emit=False, as_baseline=True)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE[args.mode], "data": "synthetic",
                "config": {"workload": "configs[1]: 0.25deg grid (145x257, dx=dy=27km), batch %d x %d query points per GPU, "
                                       "fwd + Jacobian + 6 residual terms + bwd" % (B, Np),
                           "batch_per_gpu": B, "points_per_sample": Np, "mode": args.mode,
                           "parallelism": "dp%d (samples sharded, NCCL grad all-reduce)" % world,
                           "l2": "per-step working set (%.1f GB workspace) >> 126 MB L2; no flush needed" %
                                 (Nat.workspace(Fn._shape(B, Np, 6, args.mode), dev)[1] / 2 ** 30)},
                "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu_base, "eager_gpu_baseline": eager_gpu, "clocks": clocks,
                "gpu_launches": int(holder.get("launches", 0)) * args.steps, "loss_checksum": checksum, "strong_scaling": strong,
                "other_configs": configs, "modes": modes, "sustained": sustained}
        _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
