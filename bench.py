#!/usr/bin/env python
"""bench.py -- collocation-points/sec of one loss + gradient evaluation (BASELINE.json metric).

A "step" is one pass of the hot path (pinn_loss_grad: ONE fused launch -- forward taps / residual /
reverse sweep / in-kernel gradient reduction [/ in-kernel peer-memory sum at N>1]) over the
workload's point sets.  Default workload: BASELINE.json configs[1] -- 2-D Poisson on [0,1]^2,
4x64 tanh MLP, GridTraining with 128^2 collocation points, fp32; at N>1 every rank holds a 128^2
shard of a 128 x (128 N) grid (weak scaling).  --config cfg3 | cfg4 | cfg5 runs the other BASELINE
configurations, each with its own roofline / e2e / cpu_baseline (see build_workload).

  python bench.py --gpus N --steps K --warmup W [--config cfgK]            # our engine
  python bench.py --impl reference --gpus N --steps K ... [--config cfgK]  # CPU restatement of the reference
  python bench.py ... --dump-outputs DIR     # also write the last timed step's outputs as DIR/<name>.npy

Inputs (theta, point sets) come from fixed seeds, so two builds run with the same arguments can be compared through
their dumped outputs.

Prints ONE JSON line on stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "collocation-points/sec (loss+grad)"
UNIT = "points/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Samples SM clock, power and throttle reasons during the timed region (NVML, ~2 ms period;
    falls back to nvidia-smi)."""

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        while not self._stop.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((float(clk), float(mx), {k for k, b in bits.items() if rs & b}))
            except Exception:
                pass
            self._stop.wait(0.002)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                p = [s.strip() for s in out.strip().split(",")]
                if len(p) >= 6:
                    self.rows.append((float(p[0]), float(p[1]), {n for n, v in zip(names, p[2:6]) if v.lower().startswith("active")}))
            except Exception:
                pass
            self._stop.wait(0.05)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = [r[0] for r in self.rows]
        reasons = set()
        for r in self.rows:
            reasons |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[1] for r in self.rows) if self.rows else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---- workloads: the five BASELINE.json configurations ----------------------------------------------------------------
DEFAULT_MODE = {"cfg1": "tc_split", "cfg2": "tc_split", "cfg3": "tc_bf16", "cfg4": "ffma", "cfg5": "tc_bf16"}
KERNEL_OF = {"ffma": "ffma_loss_grad_kernel", "narrow": "tc_loss_grad_kernel", "wide": "tw_loss_grad_kernel"}


def build_workload(args, world: int):
    """Config + the label both arms print.  Multi-GPU: every term's point set is sharded contiguously over the ranks.
    cfg2 weak: a 128^2 shard per rank of a 128 x 128N grid; cfg2 strong (--scaling strong): a fixed n x n grid;
    cfg3: BASELINE's 65 536 + 3 x 4 096 points (strong); cfg4: ~64^3 quadrature nodes per rank (128^3 = 2 097 152 at
    8 GPUs, as BASELINE names it); cfg5: 262 144 points per rank (1 048 576 at 4 GPUs, as BASELINE names it)."""
    from neuralpde_jl_b200 import configs
    from neuralpde_jl_b200.strategies import GridTraining
    c, n = args.config, args.n
    strong = args.scaling == "strong"
    if c == "cfg1":
        cfg = configs.config1()
        label = "1-D Poisson, 1->16->1 tanh, GridTraining 256 points (BASELINE configs[0])"
    elif c == "cfg2":
        cfg = configs.config2(n=n)
        if world > 1 and not strong:
            cfg.strategy = GridTraining([1.0 / (n - 1), 1.0 / (n * world - 1)])
        gy = n if (strong or world == 1) else n * world
        label = "2-D Poisson on [0,1]^2, 4x64 tanh MLP, GridTraining %dx%d points, fp32 (BASELINE configs[1]%s)" % (
            n, gy, "" if world == 1 else ("; sharded over %d ranks" % world if strong else "; %d-point shard per rank" % (n * n)))
    elif c == "cfg3":
        cfg = configs.config3()
        label = "2-D Burgers, 5x128 tanh MLP, 65536 stochastic collocation points + 3 x 4096 boundary points (BASELINE configs[2])"
        strong = True
    elif c == "cfg4":
        per_rank = args.points if args.points else 64 ** 3
        nodes = int(round((per_rank * (1 if strong else world)) ** (1.0 / 3.0)))
        cfg = configs.config4(nodes=nodes, bc_nodes=32)
        label = ("3-D Navier-Stokes cavity, 4 networks 3->256x6->1, fixed-node quadrature %d^3 = %d nodes x 4 equations + 19 "
                 "boundary terms x 32^2 (BASELINE configs[3]: 128^3 nodes at 8 GPUs)" % (nodes, nodes ** 3))
    elif c == "cfg5":
        per_rank = args.points if args.points else 1 << 18
        pts = per_rank * (1 if strong else world)
        cfg = configs.config5(points=pts, bcs_points=16384, n_obs=4096)
        label = ("parametric 2-D heat inverse problem (t,x,y,kappa), 4x128 tanh MLP, %d quasi-random points + 5 x 16384 "
                 "boundary points + 4096 observations, theta.p (BASELINE configs[4]: 1 048 576 points at 4 GPUs)" % pts)
    else:
        raise SystemExit("unknown config " + c)
    return cfg, label, ("strong" if strong else "weak")


def workload_sets(cfg):
    """float64 point sets [pde..., bc...] (+ quadrature weights, scales) of the workload as the CPU arm consumes them.
    Grid sets come from the oracle's own restatement of generate_training_sets (nothing of the product on the CPU arm's
    path); sampled / quadrature sets from the seeded generators the parity tests use (tests/cases.py)."""
    from neuralpde_jl_b200.strategies import GridTraining
    if isinstance(cfg.strategy, GridTraining):
        from oracle import reference as R
        sys_ = cfg.pde_system
        ps, bs = R.generate_training_sets(sys_.domain, cfg.strategy.dx, sys_.eqs, sys_.bcs, sys_.ivs, sys_.dvs)
        return ps + bs, None, None
    from cases import point_sets
    return point_sets(cfg)


def oracle_problem(cfg, derivative):
    from oracle import reference as R
    return R.Problem(cfg.pde_system, cfg.chain_specs(), param_estim=cfg.param_estim, derivative=derivative)


def cpu_reference_eval(cfg, theta64, sets, threads: int, reps: int, quad=None, derivative="fd"):
    """The reference algorithm on the host: finite-difference stencils (K forward passes per
    PDE term), mean(abs2), reverse-mode gradient, float64, all cores (oracle/reference.py)."""
    import torch
    torch.set_num_threads(threads)
    prob = oracle_problem(cfg, derivative)
    n_pde = len(cfg.pde_system.eqs)
    ps, bs = sets[:n_pde], sets[n_pde:n_pde + len(cfg.pde_system.bcs)]
    kw = {}
    if quad is not None:
        kw["qweights"], kw["qscales"] = quad
    if cfg.additional_loss is not None:
        a = cfg.additional_loss
        kw["extra"] = (1.0, prob.data_loss(a.depvar, a.points, a.values))
    times, L, G = [], None, None
    for _ in range(reps):
        t0 = time.perf_counter()
        L, _, G = prob.loss_and_grad(theta64, ps, bs, **kw)
        times.append(time.perf_counter() - t0)
    return L, times, G


def subsample(sets, quad, frac: float):
    """leading fraction of every point set (and of its quadrature weights)"""
    if frac >= 1.0:
        return sets, quad
    keep = [max(1, int(np.ceil(frac * s.shape[1]))) for s in sets]
    s2 = [s[:, :k] for s, k in zip(sets, keep)]
    q2 = None if quad is None else ([w[:k] for w, k in zip(quad[0], keep)], quad[1])
    return s2, q2


def best_thread_count(cfg, theta64, sets, quad, cores: int) -> int:
    """The reference side gets the thread count that serves it best ON THE SAMPLE IT IS TIMED ON (oversubscribing small
    GEMMs on a many-core host is slower than using fewer threads; the optimum moves with the sample size)."""
    cands = sorted({c for c in (8, 16, 32, 64) if c <= cores} or {cores})
    cpu_reference_eval(cfg, theta64, sets, cands[0], 1, quad)          # warm-up (allocator, MKL thread pool)
    best, best_t = cands[0], float("inf")
    for c in cands:
        _, t, _ = cpu_reference_eval(cfg, theta64, sets, c, 1, quad)
        if t[0] < best_t:
            best, best_t = c, t[0]
        if t[0] > 1.5 * best_t:
            break                                                       # past the optimum
    return best


def timed_cpu_sample(cfg, theta64, sets, quad, budget_s: float, reps: int):
    """Bounded sample of the workload for the CPU arm: a probe on a small leading fraction sizes the fraction that fits
    `budget_s` seconds for `reps` evaluations; the thread count is then chosen on that sample."""
    cores_all = os.cpu_count() or 1
    probe_s, probe_q = subsample(sets, quad, min(1.0, max(1.0 / 64, 2048.0 / max(s.shape[1] for s in sets))))
    cpu_reference_eval(cfg, theta64, probe_s, min(16, cores_all), 1, probe_q)
    _, tp, _ = cpu_reference_eval(cfg, theta64, probe_s, min(16, cores_all), 1, probe_q)
    n_probe = sum(s.shape[1] for s in probe_s)
    n_full = sum(s.shape[1] for s in sets)
    per_pt = tp[0] / n_probe
    frac = min(1.0, budget_s / max((reps + 5) * per_pt * n_full, 1e-9))
    s2, q2 = subsample(sets, quad, frac)
    cores = best_thread_count(cfg, theta64, s2, q2, cores_all)
    return cores, s2, q2


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    import torch  # noqa: F401
    cfg, label, scaling = build_workload(args, world)
    sets, qw, qs = workload_sets(cfg)
    quad = None if qw is None else (qw, qs)
    n_pde = len(cfg.pde_system.eqs)
    n_pts_full = sum(s.shape[1] for s in sets[:n_pde])
    if world > 1:
        # one CPU host stands beside N GPUs: it is timed on rank 0's shard (the per-rank work of the GPU arm), so its
        # points/s does not depend on N and the driver's ratio reads "N GPUs against one host"
        from neuralpde_jl_b200.strategies import shard_range
        cut = [shard_range(s.shape[1], 0, world) for s in sets]
        sets = [s[:, lo:hi] for s, (lo, hi) in zip(sets, cut)]
        if quad is not None:
            quad = ([w[lo:hi] for w, (lo, hi) in zip(quad[0], cut)], quad[1])
    theta = cfg.init_params(np.float64)
    cores, s2, q2 = timed_cpu_sample(cfg, theta, sets, quad, 150.0, args.steps + 1)
    n_pts = sum(s.shape[1] for s in s2[:n_pde])
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_reference_eval(cfg, theta, s2, cores, 1, q2)
    L, times, G = cpu_reference_eval(cfg, theta, s2, cores, args.steps, q2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"loss": np.array([L]), "grad": G})
    total = float(np.sum(times))
    val = n_pts * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": label, "n_pde_points": n_pts, "loss": L,
                   "note": "CPU host timed on %s" % ("the whole workload" if world == 1 else "rank 0's shard of it (1/%d)" % world)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d loss+grad evaluations over %d of the workload's %d PDE points (+ the same "
                                   "fraction of every other term's set); CPU restatement of the reference algorithm (FD "
                                   "stencils, PyTorch-CPU float64, best thread count), not Julia"
                                   % (args.steps, n_pts, n_pts_full)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir: str, arrays):
    """Write each array as out_dir/<name>.npy in the dtype it was computed in (float32 on the GPU, float64 on the CPU
    arm), so that two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a))


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist
    import neuralpde_jl_b200 as npde

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg, label, scaling = build_workload(args, world)
    mode = args.mode or DEFAULT_MODE[args.config]
    dtype = np.float32
    disc = cfg.discretization(dtype=dtype, mode=mode, device=local_rank)
    rep = npde.symbolic_discretize(cfg.pde_system, disc, rank=rank, world=world)
    eng = rep.engine
    n_pde = len(cfg.pde_system.eqs)
    if world > 1:
        uid = [npde.Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], rank, world)
    fused_p2p, p2p_why = eng.comm_info() if world > 1 else (False, "")

    theta_h = rep.flat_init_params
    n_theta, n_terms = eng.n_theta, eng.n_terms
    if hasattr(rep.strategy, "points") and rep.point_sets[0] is None:
        rep.loss_functions.full_loss_function(theta_h)       # Stochastic / QuasiRandom: draws + uploads the (fixed) sample
    n_pts_global = sum(rep.point_sets[i].shape[1] for i in range(n_pde))
    if world > 1 and isinstance(rep.strategy, npde.StochasticTraining):
        n_pts_global = rep.strategy.points * n_pde          # host-drawn shards: point_sets holds this rank's part
    n_other = sum(p.shape[1] for p in rep.point_sets[n_pde:] if p is not None)
    theta_d = torch.from_numpy(theta_h).to(dev)
    grad_d = torch.empty(n_theta, dtype=torch.float32, device=dev)
    terms_d = torch.empty(n_terms, dtype=torch.float32, device=dev)
    total_d = torch.empty(1, dtype=torch.float32, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MiB > 126 MB L2
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        eng.loss_grad_device(theta_d, grad_d, terms_d, total_d, None, stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        step()
    barrier()

    # ---- device-resident timing: K steps, each bracketed by CUDA events, L2 flushed between steps ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in ev:
        flush.zero_()
        a.record()
        step()
        b.record()
    barrier()
    launches = eng.launch_count() - launches0
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    t_total = float(ms.sum()) * 1e-3
    loss_val = float(total_d.item())
    grad_h = grad_d.cpu().numpy().astype(np.float64)
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the measurements below overwrite the buffers (the gradient and the
        # losses are already summed over the ranks, so rank 0 holds what every rank holds)
        dump_outputs(args.dump_outputs, {"loss": total_d.cpu().numpy(), "term_losses": terms_d.cpu().numpy(),
                                         "grad": grad_d.cpu().numpy()})

    # ---- main-kernel duration (for the roofline), events inside the library around the fused kernel ----
    eng.set_timing(True)
    kms = []
    for _ in range(min(args.steps, 20)):
        flush.zero_()
        step()
        kms.append(eng.last_kernel_ms())
    eng.set_timing(False)
    kernel_ms = float(np.mean(kms))

    # ---- end to end through host buffers (H2D theta, D2H grad + losses inside the timed region) ----
    for _ in range(3):
        eng.loss_grad_host(theta_h, None, True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tot_h, _, _ = eng.loss_grad_host(theta_h, None, True)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None

    if world > 1:
        tt = torch.tensor([t_total, t_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_total, t_e2e = float(tt[0]), float(tt[1])

    if rank == 0:
        pk, pk_kind = peaks()
        flops = eng.flops_per_eval()                                   # per-rank launch
        achieved = flops / (kernel_ms * 1e-3) / 1e12
        value = n_pts_global * args.steps / t_total
        wide = mode != "ffma" and max(max(c.dims[1:-1]) for c in cfg.chains) > 64
        kernel = KERNEL_OF["ffma" if mode == "ffma" else ("wide" if wide else "narrow")]
        tensor_bound = mode != "ffma"
        peak = pk["bf16_tflops"] if tensor_bound else 74.0            # fp32 FMA: 148 SMs x 128 lanes x 2 x 1.965 GHz
        # DRAM traffic of the dominant kernel: measured once per round with `ncu --set full` (profiles/), not re-measured here
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as fh:
                ent = json.load(fh).get("%s_%s_n%d" % (args.config, mode, args.n))
            if ent and world == 1:
                traffic, traffic_src = int(ent["dram_bytes_read"]) + int(ent["dram_bytes_write"]), ent["source"]
        except (OSError, ValueError, KeyError):
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": label, "n_pde_points": n_pts_global, "n_other_points_this_rank": n_other,
                       "mode": mode, "l2": "flushed between timed steps (256 MiB memset)",
                       "parallelism": "dp%d" % world, "loss": loss_val, "n_theta": n_theta,
                       "grad_sum": {"where": "inside the fused kernel (peer memory over NVLink)" if fused_p2p else
                                    ("ncclAllReduce" if world > 1 else "inside the fused kernel (one GPU)"),
                                    "fallback_reason": p2p_why}},
            "clocks": clocks,
            "e2e": {"value": n_pts_global * args.steps / t_e2e, "unit": UNIT,
                    "h2d_bytes_per_step": int(n_theta * 4), "d2h_bytes_per_step": int((n_theta + n_terms + 1) * 4),
                    "ms_per_step": 1e3 * t_e2e / args.steps, "api": "pinn_loss_grad_host"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor" if tensor_bound else "fp32-fma", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes (DRAM read + write per launch, ncu)",
                         "traffic_source": traffic_src, "peak_source": pk_kind if tensor_bound else "nominal fp32 FMA",
                         "kernel": kernel,
                         "arithmetic": {"ffma": "fp32 FMA on CUDA cores", "tc_bf16": "tcgen05 bf16 x bf16 -> fp32",
                                        "tc_split": "tcgen05 split-bf16 (3 MMAs per product in the forward sweep)"}[mode],
                         "kernel_ms": kernel_ms, "flops_per_launch": flops,
                         "note": "algorithmic FLOPs 6*C*S per point (SURVEY 8(d)) / fused-kernel duration (the kernel "
                                 "includes the in-kernel gradient reduction%s)" % (" and peer sum" if fused_p2p else "")},
        }
        if world == 1 and args.config == "cfg2" and not args.no_alt_modes:
            # the other arithmetic modes on the same workload (device-resident), for context
            alt = {}
            for m in ("ffma", "tc_bf16", "tc_split"):
                if m == mode:
                    continue
                d2 = cfg.discretization(dtype=dtype, mode=m, device=local_rank)
                r2 = npde.symbolic_discretize(cfg.pde_system, d2)
                for _ in range(3):
                    r2.engine.loss_grad_device(theta_d, grad_d, terms_d, total_d, None, stream)
                e2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
                for a, b in e2:
                    flush.zero_()
                    a.record()
                    r2.engine.loss_grad_device(theta_d, grad_d, terms_d, total_d, None, stream)
                    b.record()
                torch.cuda.synchronize()
                ms2 = float(np.mean([a.elapsed_time(b) for a, b in e2]))
                alt[m] = {"ms_per_step": ms2, "value": n_pts_global / (ms2 * 1e-3), "loss": float(total_d.item())}
                r2.engine.close()
            line["config"]["other_modes"] = alt
        if world == 1 and not args.no_cpu_baseline:
            sets, qw, qs = workload_sets(cfg)
            if isinstance(rep.strategy, (npde.StochasticTraining, npde.QuasiRandomTraining)):
                sets = [np.asarray(p[:len(cfg.pde_system.ivs)], dtype=np.float64) for p in rep.point_sets[:n_pde + len(cfg.pde_system.bcs)]]
            quad = None if qw is None else (qw, qs)
            th64 = theta_h.astype(np.float64)
            cores, s2, q2 = timed_cpu_sample(cfg, th64, sets, quad, 20.0, 4)
            cpu_reference_eval(cfg, th64, s2, cores, 1, q2)
            Lc, times, _ = cpu_reference_eval(cfg, th64, s2, cores, 3, q2)
            n_s = sum(s.shape[1] for s in s2[:n_pde])
            line["cpu_baseline"] = {
                "value": n_s / float(np.median(times)), "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "3 loss+grad evaluations (median) over %d of the workload's %d PDE points (+ the same fraction of "
                          "every other term's set); CPU restatement of the reference algorithm (FD stencils, PyTorch-CPU "
                          "float64, best of 8/16/32/64/all threads), not Julia" % (n_s, n_pts_global),
                "host_cores": os.cpu_count()}
            # parity of this very run against the float64 oracle (exact-tap mode) when the whole workload fits the time budget
            if args.config in ("cfg1", "cfg2", "cfg3"):
                Lx, _, Gx = cpu_reference_eval(cfg, th64, sets, cores, 1, quad, derivative="exact")
                line["cpu_baseline"]["loss"] = Lx
                line["cpu_baseline"]["loss_rel_err_engine"] = abs(loss_val - Lx) / abs(Lx)
                line["cpu_baseline"]["grad_rel_err_engine"] = float(np.linalg.norm(grad_h - Gx) / np.linalg.norm(Gx))
                if n_s == n_pts_global:
                    line["cpu_baseline"]["loss_fd"] = Lc
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configuration (cfg2 = configs[1], the headline)")
    ap.add_argument("--mode", default=os.environ.get("PINN_BENCH_MODE") or None, choices=["ffma", "tc_bf16", "tc_split"],
                    help="arithmetic mode (default: cfg2 tc_split, cfg3 / cfg5 tc_bf16, cfg4 ffma)")
    ap.add_argument("--n", type=int, default=128, help="cfg2: grid points per axis (128 = BASELINE configs[1])")
    ap.add_argument("--points", type=int, default=0, help="cfg4 / cfg5: PDE points per rank (default 64^3 / 2^18)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt-modes", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, term_losses, grad) as DIR/<name>.npy")
    args = ap.parse_args()
    # stdout carries exactly one JSON line: NCCL's version banner / debug output (printed to stdout when NCCL_DEBUG is
    # set in the environment) goes to stderr instead
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"      # NCCL honours NCCL_DEBUG_FILE only above the VERSION level
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
