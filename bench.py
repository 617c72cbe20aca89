#!/usr/bin/env python
"""bench.py -- benchmark of the batched differentiable iLQR/MPC path.

Metric (BASELINE.json): MPC solves/sec (forward + implicit backward), cartpole
T=50, B=65536 per GPU, FP64; % of the HBM roofline.

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA)
  python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on host CPU
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic problems: an
iLQR solve followed by one backward pass (the il_exp step: tile the cost, solve,
imitation loss, implicit gradient to theta, q, p).  `value` is measured with every
input resident in HBM; `e2e` is the same metric through the reference-facing API with
HOST inputs (x_init, expert controls, q, p, theta in pinned memory; the cost tensors are
tiled on the device exactly as il_env.IL_Env.mpc does; loss + gradients are copied
back).  Problems shard across GPUs by batch index with no data-path collective.

Regimes (BASELINE.md section 4, SURVEY 8d config 2):
  --regime 2a  (default, the headline) cold start, perturbation 0.5, lqr_iter = 10 fixed
               (the reference never converges there: L = 10 deterministically);
  --regime 2b  warm-started converged steady state (perturbation 0.05, u_init from an
               untimed 250-iteration pre-solve): the solve stops after one iteration and
               the implicit gradient is well posed; the line also reports how many
               Richardson passes 1e-10 needs there.
Other workloads of BASELINE.json `configs` (parity cases, each prints its own line):
  --config rocket   rocket env_dx, T=100, B=16384, box +-20, forward solves
  --config lindx    synthetic LinDx/QuadCost (--ns --nc --horizon --batch --boxed), forward + KKT backward
  --scaling strong  global batch fixed (--batch), split over the ranks
"""
import argparse
import importlib
import json
import os
import shutil
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_H = 50
NS, NC = 5, 1
N = NS + NC
LQR_ITER = 10
THETA = (9.8, 1.0, 0.1, 0.5)
METRIC = "MPC solves/sec (fwd+implicit bwd), cartpole T=50 B=64k"
# the unmodified reference's own forward (mpc_explicit.MPC, fp64, 8 host threads), measured
# in the build container where /root/reference lives (BASELINE.md section 2; it cannot travel)
REFERENCE_OWN_FORWARD = {"B=256": 134, "B=1024": 256, "B=4096": 80, "unit": "solves/s",
                         "what": "forward only, cartpole T=50 lqr_iter=10, unmodified reference "
                                 "on 8 host threads of the build container (BASELINE.md s.2)"}


def bytes_per_solve(s, L=LQR_ITER, T=T_H, n=N, ns=NS, nc=NC, ntheta=4):
    """SURVEY 8d ALGORITHMIC bytes: L fused iterations + one backward pass."""
    it = s * (T * n * n + 2 * T * n + T * nc + ns + 2)
    bwd = s * (2 * T * n * n + 4 * T * n + ns + ntheta)
    return it, bwd, L * it + bwd


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(
                    ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                     "--format=csv,noheader,nounits"], capture_output=True, text=True,
                    timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def make_inputs(torch, B, dtype, seed, sigma=0.5):
    """SURVEY 8d config 2: x,dx,dth ~ U(-s,s), th ~ U(-s,s) rad, seeded on CPU in fp64."""
    g = torch.Generator().manual_seed(seed)
    r = (torch.rand(B, 4, generator=g, dtype=torch.float64) * 2 - 1) * sigma
    x0 = torch.stack((r[:, 0], r[:, 1], torch.cos(r[:, 2]), torch.sin(r[:, 2]), r[:, 3]), 1)
    uexp = torch.randn(T_H, B, NC, generator=g, dtype=torch.float64)
    return x0.to(dtype), uexp.to(dtype)


def dump_outputs(out_dir, flat):
    """What the caller of the timed step receives (ImitationStep.run_resident: the gradients of
    the imitation loss wrt theta, q, p and the loss, summed over the ranks) as <name>.npy in
    the step's dtype; the inputs are seeded, so two builds can be compared output for output."""
    import numpy as np
    v = flat.detach().cpu().numpy()
    nth = len(THETA)
    assert v.shape == (nth + 2 * N + 1,), v.shape
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("dtheta", v[:nth]), ("dq", v[nth:nth + N]), ("dp", v[nth + N:nth + 2 * N]),
                    ("loss", v[nth + 2 * N:])):
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------ live DRAM traffic
NCU_CHILD_SKIP = 12     # launches of the dominant kernel before the captured one (warm)


def ncu_child(args):
    """Forward solves only, for the DRAM-traffic capture of the dominant kernel."""
    import torch
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    il = importlib.import_module("differentiable-ilqr_b200.il")
    dev = torch.device("cuda", 0)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    x0, uexp = make_inputs(torch, args.batch, dtype, 0, 0.5)
    step = il.ImitationStep(env.CartpoleDx, T=T_H, lqr_iter=LQR_ITER, dtype=dtype, device=dev,
                            n_richardson=1)
    q, p = [t.to(dtype).to(dev) for t in env.CartpoleDx().get_true_obj()]
    res = step.prepare(x0.to(dev), q, p, torch.tensor(THETA, dtype=dtype, device=dev))
    for _ in range(2):
        step.run_resident(res, uexp.to(dev))
    torch.cuda.synchronize()


def live_traffic(args):
    """dram__bytes_read + dram__bytes_write of ONE launch of the dominant kernel, captured
    now with ncu on a child process running the same workload (a profiler metric by nature:
    nothing timed comes from that run).  Falls back to the committed capture."""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    fallback = os.path.join(ROOT, "profiles", "r2_iter_traffic.json")
    try:
        if not os.path.exists(ncu) or args.no_ncu:
            raise RuntimeError("ncu not used")
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control",
               "none", "--print-units", "base", "--kernel-name", "regex:ilqr_iter_kernel",
               "--launch-skip",
               str(NCU_CHILD_SKIP), "--launch-count", "2", "--csv", sys.executable,
               os.path.abspath(__file__), "--ncu-child", "--dtype", args.dtype, "--batch",
               str(args.batch)]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240).stdout
        # an iteration enqueues the (symmetric, general) kernel pair and one of the two exits at
        # once (csrc/ilqr_kernels.cuh, kSym): capture two consecutive launches, keep the working one
        unit_scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        per_launch, n = {}, 0
        for line in out.splitlines():
            if "dram__bytes_" in line:
                f = [c.strip('"') for c in line.split('","')]
                per_launch[f[0]] = per_launch.get(f[0], 0.0) + \
                    float(f[-1].replace(",", "")) * unit_scale.get(f[-2], 1.0)
                n += 1
        if n != 4 or len(per_launch) != 2:
            raise RuntimeError("ncu output not understood")
        return max(per_launch.values()), \
            "ncu, this run (the working launch of one iteration, after %d warm launches)" % NCU_CHILD_SKIP
    except Exception as e:   # noqa: BLE001
        if args.dtype == "f64" and os.path.isfile(fallback):
            with open(fallback) as f:
                d = json.load(f)
            return d["dram_bytes_read"] + d["dram_bytes_write"], \
                "profiles/r2_iter_traffic.json (live capture unavailable: %s)" % str(e)[:60]
        return None, "unavailable (%s)" % str(e)[:60]


# ------------------------------------------------------------------ CUDA arm
def dist_setup(torch):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return dist, rank, world, local, dev


def make_timed(torch, dist, world, dev):
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms
    return barrier, timed


def build_step(torch, env, il, args, dtype, dev, rank, B, sigma):
    """Inputs + the il_exp-shaped step for one (dtype, regime)."""
    x0_h, uexp_h = make_inputs(torch, B, dtype, seed=rank, sigma=sigma)
    x0_h, uexp_h = x0_h.pin_memory(), uexp_h.pin_memory()
    theta_h = torch.tensor(THETA, dtype=dtype).pin_memory()
    step = il.ImitationStep(env.CartpoleDx, T=T_H, lqr_iter=LQR_ITER, dtype=dtype, device=dev,
                            n_richardson=args.richardson, tile=not args.broadcast_cost)
    q_h, p_h = [t.to(dtype).pin_memory() for t in env.CartpoleDx().get_true_obj()]
    x0, uexp = x0_h.to(dev), uexp_h.to(dev)
    res = step.prepare(x0, q_h.to(dev), p_h.to(dev), theta_h.to(dev))
    extra = {}
    if args.regime == "2b":
        # untimed pre-solve: the controls the timed solves are warm-started from
        d = importlib.import_module("differentiable-ilqr_b200")
        proto = env.CartpoleDx()
        kw = dict(u_lower=proto.lower, u_upper=proto.upper, verbose=-1, exit_unconverged=False,
                  detach_unconverged=False, linesearch_decay=proto.linesearch_decay,
                  max_linesearch_iter=proto.max_linesearch_iter, eps=proto.mpc_eps, n_batch=B)
        cost = d.QuadCost(torch.diag(q_h.to(dev)), p_h.to(dev))
        dxm = env.CartpoleDx(theta_h.to(dev))
        with torch.no_grad():
            _, u_warm, _ = d.mpc_explicit.MPC(NS, NC, T_H, lqr_iter=250, **kw)(x0, cost, dxm)
            _, u_next, _ = d.mpc_explicit.MPC(NS, NC, T_H, lqr_iter=1, u_init=u_warm, **kw)(x0, cost, dxm)
        # ~6 % of the draws end in a limit cycle of the 2-step line search instead of a fixed
        # point (there the implicit gradient does not exist and the Richardson iteration
        # diverges); the reference's own mask cannot single them out at this batch size
        # (its ||du|| rows mix 50 problems each, lqr_step.py:243-245).  Regime 2b is the
        # steady state: the batch is made of the problems that ARE at a fixed point.
        du = (u_next - u_warm).pow(2).sum((0, 2)).sqrt()
        good = (du < 1e-2 * proto.mpc_eps).nonzero().flatten()
        extra["fraction_at_fixed_point"] = good.numel() / B
        idx = good[torch.arange(B, device=dev) % good.numel()]
        x0, uexp, u_warm = x0[idx].contiguous(), uexp[:, idx].contiguous(), u_warm[:, idx].contiguous()
        x0_h, uexp_h = x0.cpu().pin_memory(), uexp.cpu().pin_memory()
        res = step.prepare(x0, q_h.to(dev), p_h.to(dev), theta_h.to(dev))
        step.mpc.u_init = u_warm
        # how many Richardson passes does 1e-10 take at this point?
        probe = il.ImitationStep(env.CartpoleDx, T=T_H, lqr_iter=LQR_ITER, dtype=dtype, device=dev,
                                 n_richardson=30, richardson_tol=1e-10, tile=not args.broadcast_cost)
        probe.mpc.u_init = u_warm
        probe.defer = False
        probe.run_resident(res, uexp)
        extra["richardson_passes_for_1e-10"] = probe.mpc.last_backward.get("passes")
        extra["richardson_residual_reached"] = probe.mpc.last_backward.get("resid")
    return step, res, (x0_h, uexp_h, q_h, p_h, theta_h), uexp, extra


def run_b200(args):
    import torch
    lib = importlib.import_module("differentiable-ilqr_b200._lib")
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    il = importlib.import_module("differentiable-ilqr_b200.il")
    warnings.filterwarnings("ignore", message="DiLQR backward: after")   # reported in `config`
    dist, rank, world, local, dev = dist_setup(torch)
    barrier, timed = make_timed(torch, dist, world, dev)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    s = 8 if dtype == torch.float64 else 4
    strong = args.scaling == "strong"
    B = args.batch // world if strong else args.batch
    sigma = 0.5 if args.regime == "2a" else 0.05

    step, res, host, uexp, extra = build_step(torch, env, il, args, dtype, dev, rank, B, sigma)
    x0_h, uexp_h, q_h, p_h, theta_h = host

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()

    # --- value: inputs resident in HBM ------------------------------------
    lib.profile = None
    n0 = lib.launch_count
    last = {}

    def resident_step():
        last["flat"] = step.run_resident(res, uexp)
    ms = timed(resident_step, args.steps, args.warmup)
    launches = (lib.launch_count - n0) // (args.steps + args.warmup) * args.steps
    info, bstat = step.mpc.last_info, dict(step.mpc.last_backward or {})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["flat"])

    # --- per-kernel timing (CUDA events on the launching stream) -------------
    lib.profile = {}
    barrier()
    for _ in range(max(1, min(args.steps, 3))):
        step.run_resident(res, uexp)
    torch.cuda.synchronize()
    prof = {k: [a.elapsed_time(b) for a, b in v] for k, v in lib.profile.items()}
    lib.profile = None
    it_all = prof.get("dilqr_mpc_iterate", [0.0])
    # launches that did work (regime 2b: the device-side stop rule turns the rest into no-ops)
    n_live = max(1, info.n_iters) * max(1, min(args.steps, 3))
    it_ms = sorted(it_all, reverse=True)[:n_live] if args.regime == "2b" else it_all
    it_avg = sum(it_ms) / max(1, len(it_ms))

    # --- e2e: host inputs, H2D / D2H inside the timed region ---------------
    ms_e2e = timed(lambda: step.run_host(x0_h, uexp_h, q_h, p_h, theta_h), args.steps,
                   args.warmup)
    h2d = (x0_h.numel() + uexp_h.numel() + q_h.numel() + p_h.numel() + theta_h.numel()) * s
    d2h = step.d2h_bytes

    # --- the other dtype, same step (value only) ------------------------------
    other = None
    if not args.single_dtype and args.regime == "2a" and not strong:
        odt = torch.float32 if dtype == torch.float64 else torch.float64
        so = 4 if odt == torch.float32 else 8
        ostep, ores, _, ouexp, _ = build_step(torch, env, il, args, odt, dev, rank, B, sigma)
        oms = timed(lambda: ostep.run_resident(ores, ouexp), args.steps, args.warmup)
        lib.profile = {}
        ostep.run_resident(ores, ouexp)
        torch.cuda.synchronize()
        oit = [a.elapsed_time(b) for a, b in lib.profile.get("dilqr_mpc_iterate", [])]
        lib.profile = None
        oit_b, _, otot_b = bytes_per_solve(so)
        oavg = sum(oit) / max(1, len(oit))
        hbm_o, _ = peaks()
        other = {"dtype": "f32" if odt == torch.float32 else "f64", "ms_per_step": oms,
                 "value": world * B / (oms * 1e-3), "unit": "solves/s",
                 "roofline_frac_of_solve": B / (oms * 1e-3) * otot_b / (hbm_o * 1e9),
                 "iter_kernel": {"avg_launch_ms": oavg,
                                 "frac": (oit_b * B / (oavg * 1e-3) / 1e9 / hbm_o) if oavg else None}}
        del ostep, ores, ouexp
        torch.cuda.empty_cache()

    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    if rank == 0:
        hbm, which = peaks()
        L_run = info.n_iters if args.regime == "2b" else LQR_ITER
        it_b, bwd_b, tot_b = bytes_per_solve(s, L=L_run)
        achieved = it_b * B / (it_avg * 1e-3) / 1e9 if it_avg > 0 else 0.0
        value = world * B / (ms * 1e-3)
        traffic, traffic_src = (None, "not captured (broadcast cost / multi-GPU run)")
        if world == 1 and not args.broadcast_cost and args.regime == "2a":
            traffic, traffic_src = live_traffic(args)
        sname = "double" if args.dtype == "f64" else "float"
        line = {
            "metric": METRIC,
            "value": value, "unit": "solves/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": args.dtype,
            "data": "synthetic",
            "config": {
                "workload": "cartpole env_dx MPC T=50 B=%d/GPU forward(lqr_iter=10, %s)+%s backward, "
                            "per B200" % (B, "cold start sigma=0.5" if args.regime == "2a" else
                                          "warm start sigma=0.05 at a fixed point, stops after %d "
                                          "iteration(s)" % info.n_iters,
                                          step.backward_name),
                "regime": args.regime, "batch_per_gpu": B, "T": T_H, "lqr_iter": LQR_ITER,
                "iterations_run": L_run,
                "l2": "inputs larger than L2 (C alone is %.2f GB)" % (T_H * B * N * N * s / 1e9),
                "parallelism": "batch-sharded x%d, no data-path collective" % world,
                "roofline_frac_of_solve": value / world * tot_b / (hbm * 1e9),
                "bytes_per_solve": tot_b, "richardson_passes": args.richardson,
                "richardson_last_update_rel": bstat.get("resid"),
                "backward": "fused" if bstat.get("fused") else "round-1 sequence",
                "cost_layout": "broadcast [n,n]" if args.broadcast_cost else "dense [T,B,n,n]",
                "trace_retries": step.retries, "steps_redone": step.redone,
            },
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                         "frac": achieved / hbm, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": which,
                         "kernel": "ilqr_iter_kernel<%s,5,1,CARTPOLE>" % sname,
                         "algorithmic_bytes_per_launch": it_b * B,
                         "avg_launch_ms": it_avg},
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "solves/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches,
            "clocks": sampler.summary() if sampler else None,
            "kernel_ms": {k: sum(v) / len(v) for k, v in prof.items()},
        }
        line["config"].update(extra)
        if other is not None:
            line["other_dtype"] = other
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(dtype, sample_B=args.cpu_batch,
                                                n_passes=args.richardson)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ other workloads
def run_other(args):
    """--config rocket | lindx: the remaining BASELINE.json configs as bench lines."""
    import torch
    d = importlib.import_module("differentiable-ilqr_b200")
    env = importlib.import_module("differentiable-ilqr_b200.env_dx")
    dist, rank, world, local, dev = dist_setup(torch)
    barrier, timed = make_timed(torch, dist, world, dev)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    s = 8 if dtype == torch.float64 else 4
    B = args.batch // world if args.scaling == "strong" else args.batch
    g = torch.Generator().manual_seed(rank)
    hbm, which = peaks()
    if args.config == "rocket":
        T, ns, nc = args.horizon or 100, 13, 3
        dx = env.RocketDx(torch.tensor((0.5, 1.0, 1.0, 1.0, 1.0), dtype=dtype, device=dev))
        qv = torch.cat((torch.ones(B, 1, dtype=torch.float64),
                        0.1 * torch.randn(B, 3, generator=g, dtype=torch.float64)), 1)
        x0 = torch.cat(((torch.rand(B, 3, generator=g, dtype=torch.float64) * 2 - 1) * 15,
                        torch.rand(B, 3, generator=g, dtype=torch.float64) * 2 - 1,
                        qv / qv.norm(dim=1, keepdim=True),
                        (torch.rand(B, 3, generator=g, dtype=torch.float64) * 2 - 1) * 0.1), 1)
        x0 = x0.to(dtype).to(dev)
        q, p = [t.to(dtype).to(dev) for t in dx.get_true_obj()]
        C = torch.diag(q)[None, None].repeat(T, B, 1, 1)
        c = p[None, None].repeat(T, B, 1)
        m = d.mpc_explicit.MPC(ns, nc, T, u_lower=-20.0, u_upper=20.0, lqr_iter=LQR_ITER, verbose=-1,
                               exit_unconverged=False, detach_unconverged=False,
                               linesearch_decay=dx.linesearch_decay,
                               max_linesearch_iter=dx.max_linesearch_iter, eps=dx.mpc_eps, n_batch=B)

        def fn():
            with torch.no_grad():
                m(x0, d.QuadCost(C, c), dx)
        what = "rocket env_dx MPC T=%d B=%d/GPU box +-20, forward solve (lqr_iter=10)" % (T, B)
        L = None
    else:
        T, ns, nc = args.horizon or 50, args.ns, args.nc
        # SURVEY 8d config 5 generator (tests/common.lindx_problem), drawn on the device: at
        # B = 1 M the host generator alone would take minutes
        gd = torch.Generator(device=dev).manual_seed(rank)
        nn_ = ns + nc
        rn = lambda *sh: torch.randn(*sh, generator=gd, dtype=dtype, device=dev)
        A = rn(T, B, nn_, nn_)
        Cc = torch.baddbmm(torch.eye(nn_, dtype=dtype, device=dev).expand(T * B, nn_, nn_),
                           A.view(T * B, nn_, nn_).transpose(1, 2), A.view(T * B, nn_, nn_)
                           ).view(T, B, nn_, nn_)
        del A
        cc = rn(T, B, nn_)
        F = torch.cat((torch.eye(ns, dtype=dtype, device=dev).expand(T - 1, B, ns, ns)
                       + 0.2 * rn(T - 1, B, ns, ns) / ns ** 0.5,
                       rn(T - 1, B, ns, nc) / ns ** 0.5), 3).contiguous()
        f = 0.1 * rn(T - 1, B, ns)
        x0 = rn(B, ns)
        kw = dict(u_lower=-1.0, u_upper=1.0) if args.boxed else {}
        m = d.MPC(ns, nc, T, lqr_iter=LQR_ITER, verbose=-1, exit_unconverged=False,
                  detach_unconverged=False, n_batch=B, **kw)
        Cg, cg = Cc.requires_grad_(), cc.requires_grad_()

        def fn():
            Cg.grad = cg.grad = None
            x, u, _ = m(x0, d.QuadCost(Cg, cg), d.LinDx(F, f))
            (x.sum() + u.sum()).backward()
        what = ("synthetic LinDx/QuadCost ns=%d nc=%d T=%d B=%d/GPU %s, forward (lqr_iter<=10) + KKT "
                "backward" % (ns, nc, T, B, "box +-1" if args.boxed else "unconstrained"))
    n = ns + nc
    ms = timed(fn, args.steps, args.warmup)
    info = m.last_info
    L = info.n_iters
    it = s * (T * n * n + 2 * T * n + T * nc + ns + 2) + (0 if args.config == "rocket" else
                                                          s * (T - 1) * (ns * n + ns))
    bwd = 0 if args.config == "rocket" else s * (2 * T * n * n + 4 * T * n + 2 * (T - 1) * ns * n)
    tot = L * it + bwd
    if rank == 0:
        print(json.dumps({
            "metric": "MPC solves/sec, " + args.config, "value": world * B / (ms * 1e-3),
            "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if args.scaling == "strong" else "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": what, "iterations_run": L, "trace_retries": info.retries,
                       "bytes_per_solve": tot,
                       "roofline_frac_of_solve": B / (ms * 1e-3) * tot / (hbm * 1e9),
                       "peak_source": which}}))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------- reference arm
def cpu_solve_once(torch, port, dtype, B, seed=0, n_passes=4):
    """One step of the same workload with the oracle port (== the reference's
    algorithm, validated bit-exact against it) on the host CPU."""
    x0, uexp = make_inputs(torch, B, dtype, seed)
    dx = port.CartpoleDx(dtype=dtype)
    q, p = dx.get_true_obj()
    C = torch.diag(q)[None, None].repeat(T_H, B, 1, 1)
    c = p[None, None].repeat(T_H, B, 1)
    t0 = time.time()
    o = port.mpc_forward(x0, port.QuadCost(C, c), dx, NS, NC, T_H, u_lower=dx.lower,
                         u_upper=dx.upper, lqr_iter=LQR_ITER, eps=dx.mpc_eps,
                         linesearch_decay=dx.linesearch_decay,
                         max_linesearch_iter=dx.max_linesearch_iter, final_pass=True)
    gu = 2.0 * (o.u - uexp) / o.u.numel()
    gx = torch.zeros_like(o.x)
    port.dilqr_backward(gx, gu, x0, C, c, o.x, o.u, dx, NS, NC, dx.lower, dx.upper,
                        n_passes=n_passes)
    return time.time() - t0


def cpu_baseline(dtype, sample_B=2048, n_passes=4):
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import port
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    with torch.no_grad():
        dt = cpu_solve_once(torch, port, dtype, sample_B, n_passes=n_passes)
    return {"value": sample_B / dt, "unit": "solves/s", "cores": cores, "kind": "port",
            "sample": "B=%d problems of the same workload (forward lqr_iter=10 + DiLQR backward, "
                      "%d Richardson passes) with the oracle port of the reference, %.1f s"
                      % (sample_B, n_passes, dt),
            "reference_own_forward": REFERENCE_OWN_FORWARD}


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import port
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    with torch.no_grad():
        # size the sample so that W warm-up + exactly K timed steps end within ~3 minutes:
        # the port's rate is measured on a small batch first (it only grows with B)
        cpu_solve_once(torch, port, dtype, 64, n_passes=args.richardson)
        probe_B = 1024
        rate = probe_B / cpu_solve_once(torch, port, dtype, probe_B, n_passes=args.richardson)
        budget = 170.0 / (args.steps + min(args.warmup, 2) * 0.25)
        Bs = args.cpu_batch
        while Bs > 256 and Bs / rate > budget:
            Bs //= 2
        for i in range(min(args.warmup, 2)):
            cpu_solve_once(torch, port, dtype, max(64, Bs // 4), seed=100 + i, n_passes=args.richardson)
        t = [cpu_solve_once(torch, port, dtype, Bs, seed=i, n_passes=args.richardson)
             for i in range(args.steps)]
    ms = 1e3 * sum(t) / len(t)
    v = Bs / (ms * 1e-3)
    sample = ("B=%d problems per step (sized to the time budget of %d steps) on %d host threads, "
              "oracle port of the reference (its matrix-free backward; the reference's own dense "
              "fix_point_equ is limited to T*B < 1000)" % (Bs, args.steps, cores))
    print(json.dumps({
        "impl": "reference",
        "metric": METRIC,
        "value": v, "unit": "solves/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)),
        "steps": len(t), "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.dtype,
        "data": "synthetic",
        "config": {"workload": "cartpole env_dx MPC T=50 forward(lqr_iter=10, cold start sigma=0.5)"
                               "+DiLQR implicit (%d Richardson passes) backward, oracle port of "
                               "the reference on host CPU" % args.richardson, "batch": Bs},
        "cpu_baseline": {"value": v, "unit": "solves/s", "cores": cores, "kind": "port",
                         "sample": sample, "reference_own_forward": REFERENCE_OWN_FORWARD},
        "e2e": {"value": v, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of each measured loop")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before each measured loop")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dtype", default="f64", choices=["f64", "f32"])
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--cpu-batch", type=int, default=32768)
    ap.add_argument("--richardson", type=int, default=4)
    ap.add_argument("--regime", default="2a", choices=["2a", "2b"])
    ap.add_argument("--config", default="cartpole", choices=["cartpole", "rocket", "lindx"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--ns", type=int, default=8)
    ap.add_argument("--nc", type=int, default=2)
    ap.add_argument("--horizon", type=int, default=None)
    ap.add_argument("--boxed", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--single-dtype", action="store_true",
                    help="skip the second (other dtype) measurement of the same step")
    ap.add_argument("--no-ncu", action="store_true",
                    help="do not capture the dominant kernel's DRAM traffic with ncu")
    ap.add_argument("--ncu-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--broadcast-cost", action="store_true",
                    help="hand MPC the [n,n]/[n] cost (mpc.py:205-219 broadcast) instead of the "
                         "dense [T,B,n,n] tiling of il_env.py:159-162 (not the headline config)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (dtheta, dq, dp, loss) as "
                         "DIR/<name>.npy (cartpole step of the CUDA implementation)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.config != "cartpole"):
        ap.error("--dump-outputs is available for the cartpole step of --impl b200 only")
    if args.batch is None:
        args.batch = 16384 if args.config == "rocket" else 65536
    if args.ncu_child:
        ncu_child(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.config != "cartpole":
        run_other(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
