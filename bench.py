#!/usr/bin/env python
"""bench.py -- full NLP evaluations per second of the B200 evaluator (BASELINE.json metric).

One *step* = one full evaluation of one iterate of the workload problem: constraint residual +
sparse constraint Jacobian + sparse Hessian of the Lagrangian (objective and gradient are computed
in the same pass and are part of the step).  Headline workload: BASELINE.json configs[1] ("c2"):
bilinear isomorphic-state quantum gate problem, state dim 32, 4 drives, N=2000 knots, free dt +
MinimumTimeObjective.  With --gpus N > 1 every rank evaluates its own independent problem of the
same shape (problem-parallel, no data-path collective): weak scaling.

  value      whole-job evaluations/s with Z, mu and all outputs resident in HBM (dto_eval_all_dev)
  e2e        the same metric through the host-pointer C ABI as a solver calls it: the five callbacks
             (objective, gradient, constraint, Jacobian, Hessian) on a NEW iterate every step, page-locked
             host buffers, the solver's value arrays registered once (dto_register_outputs); H2D of Z and mu
             and D2H of all five outputs inside the timed region.  e2e.fused: the single dto_eval_all call.
  roofline   dominant kernel (K1, the bilinear interval kernel; K7 for c3): algorithmic FP64 flops per launch
             (SURVEY.md section 8d canonical counts) / CUDA-event duration measured live
  cpu_baseline   the CPU oracle port timed on the host cores on a bounded sample of the same workload
  extra      (default run only) the other BASELINE.json configurations at this GPU count, each a short run of
             the same measurement: c3 (TDBI, one problem per GPU), c4 (ONE trajectory in knot-range shards:
             halo and scalars through CUDA-IPC exchange windows over NVLink) and c5 (batch split), with
             `shard_matches_single_gpu`: the sharded outputs compared bit for bit with the unsharded evaluation.

`--impl reference` times the reference's CPU algorithm for the path (the oracle port; the reference
is Julia and neither Julia nor its packages exist here or on the GPU box) on the same config.
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

WORKLOADS = {
    # BASELINE.json configs[1] (the configuration the metric is quoted on): one problem per GPU, weak scaling
    "c2": dict(kind="gate", N=2000, levels=16, n_drives=4, mode="replicas"),
    # configs[2]: TimeDependentBilinearIntegrator + derivative chain + knot constraints, one problem per GPU
    "c3": dict(kind="carrier", N=1000, state_dim=64, n_drives=2, mode="replicas"),
    # configs[3]: ONE long trajectory, knot ranges sharded over the ranks with a one-knot NVLink halo (strong scaling)
    "c4": dict(kind="scaled", N=100000, state_dim=16, n_controls=2, generator_scale=0.25, mode="knot_shards"),
    # configs[4]: 4096 independent 8-state problems, problem-parallel over the ranks (strong scaling)
    "c5": dict(kind="scaled", N=200, state_dim=8, n_controls=2, generator_scale=0.35, batch=4096, mode="batch_split"),
}
FP64_PEAK_TFLOPS = 37.1  # measured on this pool's B200: DMMA m8n8k4 saturation (profiles/r01_fp64_peaks_and_box_probe.log)
TAYLOR_T = 20            # canonical term count of SURVEY.md section 8d (C1)
TDB_RHS = 80             # right-hand sides per interval of K7 with eight extrapolation columns and one macro step (BASELINE.md section 3); the kernels size the columns per interval: tdb_rhs_per_interval
DUMP_MAX_ENTRIES = 1 << 20  # per array of --dump-outputs: five float64 arrays stay under 64 MB at every workload


def dump_outputs(directory, arrays):
    """--dump-outputs: writes each output as <directory>/<name>.npy (float64, flattened).  An array of more than
    DUMP_MAX_ENTRIES entries is stored as its entries at a fixed sample of positions (seed 0, sorted), so that two builds
    run with the same arguments can be compared entry for entry."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
        if a.size > DUMP_MAX_ENTRIES:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ENTRIES, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def canonical_flops_per_interval(n, m, T=TAYLOR_T, s=0):
    """SURVEY.md section 8d, count C1: (i) full propagator by Pade-13 scaling and squaring,
    (ii) forward second-order directional propagation, (iii) adjoint first-order propagation."""
    p = m + 1
    i = 2 * n**3 * (6 + s) + (8.0 / 3.0) * n**3
    ii = (1 + 2 * p + 3 * p * (p + 1) / 2) * T * 2 * n * n
    iii = (1 + 2 * p) * T * 2 * n * n
    return i + ii + iii


def canonical_flops_per_tdb_interval(n, m, spline_order=1, rhs=TDB_RHS):
    """Count C3 (BASELINE.md section 3; SURVEY.md section 8d "the same (ii)/(iii) structure with p = 2m+2"): per
    right-hand side of the variational system, n mat-vecs for the propagator, 1 + 2p + 3p(p+1)/2 for the second-order
    forward jet and 1 + 2p for the first-order adjoint, 2 n^2 flops each; p = parameters [u_k, (u_k+1), dt, t]."""
    p = (2 * m if spline_order == 1 else m) + 2
    matvecs = n + (1 + 2 * p + 3 * p * (p + 1) / 2) + (1 + 2 * p)
    return rhs * matvecs * 2 * n * n


def tdb_rhs_per_interval(prob, Zvec):
    """Right-hand sides K7 evaluates per interval at this iterate: the host restatement of `tdb_item_steps`
    (csrc/dto_internal.h): theta = |dt| (||G0||_1 + sum ||D_j||_1 + sum_i max|u_i| (||A_i||_1 + ||B_i||_1) + max omega); ceil(theta)
    macro steps above 1; the smallest K in 3..8 columns with theta^(2K+1) <= tol (2^K K!)^2 (DTO_B200_TDB_TOL, default 1e-14;
    0: eight columns); a sweep of K columns costs sum_{k<=K} (2k + 1) = K^2 + 2K right-hand sides."""
    it = prob.integrators[0]
    t = prob.trajectory
    G = it.G
    n1 = lambda M: float(np.abs(M).sum(axis=0).max()) if M.size else 0.0
    gnorm = n1(G.G0) + sum(n1(D) for D in G.D)
    bnorm = np.array([n1(G.A[i]) + n1(G.B[i]) for i in range(G.A.shape[0])])
    wmax = float(max([0.0] + [abs(w) for w in G.omega] + [abs(w) for w in G.omega_d]))
    tol = float(os.environ.get("DTO_B200_TDB_TOL", "1e-14"))
    Zm = np.asarray(Zvec)[: t.N * t.dim].reshape(t.N, t.dim)
    u = np.abs(Zm[:, t.components[it.u_name]])
    dt = np.abs(Zm[:, t.components[t.timestep]]).reshape(t.N)
    total = 0
    for k in range(t.N - 1):
        uk = np.maximum(u[k], u[k + 1]) if it.spline_order == 1 else u[k]
        theta = dt[k] * (gnorm + float(uk @ bnorm) + wmax)
        steps = max(1, int(it.steps) if it.steps else 1)
        if theta > steps:
            steps = min(256, int(np.ceil(theta)))
        K = 8
        if tol > 0:
            ths, den = theta / steps, 2304.0
            for kk in range(3, 8):
                if ths ** (2 * kk + 1) <= tol * den:
                    K = kk
                    break
                den *= 4.0 * (kk + 1) ** 2
        total += steps * (K * K + 2 * K)
    return total / max(1, t.N - 1)


def recorded_traffic(workload, variant):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the committed
    `ncu --set full` capture of this workload and kernel variant (profiles/); None when no capture matches."""
    for rnd in ("r02", "r01"):
        path = os.path.join(ROOT, "profiles", f"{rnd}_ncu_summary_{workload}.json")
        try:
            full = json.load(open(path))["k1_ncu_set_full"]
            if variant in full["kernel"]:
                return float(full["dram_bytes_per_launch"]), os.path.relpath(path, ROOT)
        except Exception:
            pass
    return None, None


def build_problem(workload, seed):
    import dto_b200 as dto

    kw = dict(WORKLOADS[workload])
    kind = kw.pop("kind")
    kw.pop("batch", None)
    kw.pop("mode", None)
    if kind == "gate":
        return dto.problem_templates.quantum_gate_problem(seed=seed, **kw)
    if kind == "carrier":
        return dto.problem_templates.carrier_problem(seed=seed, **kw)
    return dto.problem_templates.scaled_problem(seed=seed, **kw)


def workload_config(workload, prob, mode):
    """The `config` both arms print (identical strings: the driver pairs the two lines by it)."""
    t = prob.trajectory
    n, m, z, N = t.dims["x"], t.dims["u"], t.dim, t.N
    dsum = sum(i.x_dim for i in prob.integrators)
    rows, jac = (N - 1) * dsum, (N - 1) * dsum * 2 * z
    hess = N * z * (z + 1) // 2 + (N - 1) * z * z
    batch = WORKLOADS[workload].get("batch")
    what = {"c2": "bilinear quantum gate", "c3": "time-dependent bilinear (carrier drives, linear spline) + derivative chain + norm(u) <= 1",
            "c4": "random dense bilinear (make_scaled_problem)", "c5": "random dense bilinear (make_scaled_problem)"}[workload]
    return {
        "workload": f"{workload}: {what}, state dim {n}, {m} drives, N={N}" + (f", batch {batch}" if batch else "") +
                    f" (z={z}; per problem: {N * z} vars, {rows} dynamics rows, {jac} dynamics Jac nnz, {hess} Hess nnz)",
        "per_rank": {"replicas": "one independent problem per GPU (problem-parallel, no collective)",
                     "knot_shards": "contiguous knot range of ONE trajectory per GPU; every step uploads a new iterate, pushes the shard's first knot into the left "
                                    "neighbour's CUDA-IPC exchange window (NVLink P2P) and reduces objective + violation through the same windows (one kernel, no NCCL)",
                     "batch_split": "contiguous block of the problem batch per GPU (no collective)"}[mode],
        "step": "objective+gradient+constraint+Jacobian+Hessian of one iterate",
    }


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons while the timed region runs: NVML in-process (a query takes ~50 us, so even a
    few-millisecond region gets several samples; one `nvidia-smi` process start takes longer than the whole region), the
    `nvidia-smi` query line of the profiling recipe as fallback."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows, self.source = index, threading.Event(), [], "nvml"
        self.nv = self.handle = None
        try:
            import pynvml as nv
            import torch

            nv.nvmlInit()
            try:  # the CUDA device of this rank, whatever the enumeration order
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.handle = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = nv.nvmlDeviceGetHandleByIndex(index)
            self.nv = nv
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            self.source = "nvidia-smi"

    def _nvml_row(self):
        nv = self.nv
        mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
        get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        r = int(get(self.handle))
        bits = [getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8), getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20), getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)]
        return [str(mhz), str(self.max_mhz)] + ["Active" if r & b else "Not Active" for b in bits]

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                if self.nv is not None:
                    self.rows.append(self._nvml_row())
                else:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.002 if self.nv is not None else 0.02)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = [n for i, n in enumerate(self.NAMES) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "source": self.source}


def cpu_port_rate(prob, sample_intervals, threads, all_dirs=True):
    """Oracle port timed on the host: full constraint+Jacobian+Hessian work of `sample_intervals`
    knot intervals (the reference's cost is linear in N: serial knot loop,
    src/integrators/bilinear_integrator.jl:99,113,142), scaled to evaluations/s of the whole problem."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dto_oracle_c as oc

    return oc.time_port(prob, sample_intervals, threads, all_dirs=all_dirs)


def run_reference(args, rank, world):
    if rank != 0:
        return
    workload = "c2" if args.workload == "all" else args.workload
    if workload == "c3":
        print(json.dumps({"impl": "reference", "unavailable": "the C port of the reference algorithm covers BilinearIntegrator only (c2, c4, c5)"}), flush=True)
        return
    prob = build_problem(workload, seed=42)
    threads = os.cpu_count() or 1
    vals = []
    sample = args.ref_sample
    for i in range(args.warmup + args.steps):
        rate, info = cpu_port_rate(prob, sample, threads)
        if i >= args.warmup:
            vals.append(rate)
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": "full NLP evals/sec (constraint+Jacobian+Hessian)", "value": v, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(workload, prob, WORKLOADS[workload]["mode"]),
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": info["threads"], "kind": "port", "sample": info["sample"]},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # machine-readable: the number is a linear extrapolation from a sample of the intervals, not a timed whole evaluation
        "extrapolated": True, "extrapolation": {"timed_intervals": int(min(sample, prob.trajectory.N - 1)), "of_intervals": prob.trajectory.N - 1,
                                                "rule": "seconds per interval x (N - 1): the reference's knot loop is serial"},
        "note": "reference is Julia (absent here and on the GPU box); this arm times oracle/dto_oracle.c, a C restatement of the reference's ForwardDiff-through-expv algorithm, POSIX threads over knot intervals, all host cores",
    }
    print(json.dumps(line), flush=True)


def run_workload(args, workload, steps, warmup, *, rank, world, local_rank, full):
    """One measurement of one workload on this rank; returns (on rank 0) the JSON line as a dict.
    `full`: the headline line (cpu_baseline, fused e2e, clocks); otherwise the short `extra` form."""
    import torch
    import torch.distributed as dist

    import dto_b200 as dto
    from dto_b200.sharding import ShardedEvaluator, split_batch

    mode = WORKLOADS[workload]["mode"]
    prob = build_problem(workload, seed=42 + (rank if mode == "replicas" else 0))
    t = prob.trajectory
    n, m = t.dims["x"], t.dims["u"]
    rng = np.random.default_rng(1234 + rank)
    sharded = None
    batch_local = 1
    if mode == "replicas":  # an independent problem per rank
        ev = dto.Evaluator(prob, device=local_rank)
        Z = t.datavec.copy()
    elif mode == "knot_shards":
        sharded = ShardedEvaluator(prob, rank, world, device=local_rank, dist=dist if world > 1 else None)
        ev = sharded.local
        Z = sharded.local_slice(t.datavec)
    else:
        B = WORKLOADS[workload]["batch"]
        b0, b1 = split_batch(B, world)[rank]
        batch_local = b1 - b0
        ev = dto.Evaluator(prob, device=local_rank, batch=batch_local)
        Z = np.tile(t.datavec, batch_local) + 0.01 * np.random.default_rng(77).standard_normal((B, ev.n_vars))[b0:b1].reshape(-1)
    mu = rng.random(batch_local * ev.n_constraints)
    sigma = 1.0
    n_grad = batch_local * (ev.shard_layout.z_end - ev.shard_layout.z_begin)
    linked = sharded is not None and world > 1

    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.ExternalStream(ev.stream, device=dev)
    # two device-resident iterates in rotation: a sharded step uploads (device to device) and publishes a new one every time
    dZs = [torch.from_numpy(Z).to(dev), torch.from_numpy(Z + 1e-3 * rng.standard_normal(Z.size)).to(dev)]
    dmu = torch.from_numpy(mu).to(dev)
    dJ = torch.empty(batch_local, dtype=torch.float64, device=dev)
    dviol = torch.zeros(batch_local, dtype=torch.float64, device=dev)
    dgrad = torch.empty(n_grad, dtype=torch.float64, device=dev)
    dg = torch.empty(batch_local * ev.n_constraints, dtype=torch.float64, device=dev)
    djac = torch.empty(batch_local * ev.nnz_jacobian, dtype=torch.float64, device=dev)
    dhess = torch.empty(batch_local * ev.nnz_hessian, dtype=torch.float64, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)  # > 126 MB L2
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()

    def step_dev(i):
        zp = dZs[i % 2].data_ptr()
        if sharded is not None:
            # the shard's iterate lives in the evaluator's own buffer; upload_dev copies the new iterate there and pushes
            # this shard's first knot into the left neighbour's exchange window (NVLink P2P)
            ev.upload_dev(zp)
            zp = ev.local_Z_ptr
        ev.eval_all_dev(zp, sigma, dmu.data_ptr(), dJ.data_ptr(), dgrad.data_ptr(), dg.data_ptr(), djac.data_ptr(), dhess.data_ptr())
        if linked:
            # the only exchange of the sharded path besides the halo knot: objective (sum) and violation (max)
            if args.scalar_reduce == "peer":  # violation of the shard's rows + exchange through the peer windows: one kernel
                ev.shard_scalars_dev(dg.data_ptr(), dJ.data_ptr(), dviol.data_ptr())
            else:
                ev.violation_dev(dg.data_ptr(), dviol.data_ptr())
                dist.all_reduce(dJ, op=dist.ReduceOp.SUM)
                dist.all_reduce(dviol, op=dist.ReduceOp.MAX)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ------------------------------------------------------------------
    with torch.cuda.stream(stream):
        for i in range(warmup):
            flush.zero_()
            step_dev(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if full:
        sampler.start()
    l0 = ev.launch_count
    ev.kernel_timing(True)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    t_wall0 = time.perf_counter()
    with torch.cuda.stream(stream):
        for i, (e0, e1) in enumerate(evs):
            flush.zero_()  # L2 flush between timed iterations (outside the per-step events)
            e0.record(stream)
            step_dev(i)
            e1.record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    if full:  # the clocks of the device-timed region are sampled; the host-path timing below runs without the sampler thread
        sampler.stop_flag.set()
        sampler.join()
    step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    k1_ms, k1_n = ev.kernel_time_ms()
    ev.kernel_timing(False)
    launches = ev.launch_count - l0
    dev_ms = float(np.sum(step_ms))
    if args.dump_outputs and full and rank == 0:  # what the last timed step left in HBM, before anything overwrites it
        dump_outputs(args.dump_outputs, {"objective": dJ.cpu().numpy(), "gradient": dgrad.cpu().numpy(), "constraint": dg.cpu().numpy(),
                                         "jacobian": djac.cpu().numpy(), "hessian": dhess.cpu().numpy()})
    # outputs of iterate 0 for the parity guards below
    with torch.cuda.stream(stream):
        step_dev(0)
    barrier()
    ref_out = [x.cpu().numpy() for x in (dg, djac, dhess)]
    J_total = float(dJ[0].item())

    # ---- sharded == unsharded, bit for bit -------------------------------------------------------
    shard_ok = None
    if mode == "knot_shards" and world > 1:
        whole = dto.Evaluator(prob, device=local_rank)
        wz = torch.from_numpy(t.datavec.copy()).to(dev)
        rows, jpos, hpos = ev.shard_maps()
        wmu = torch.zeros(whole.n_constraints, dtype=torch.float64, device=dev)
        wmu[torch.from_numpy(rows).to(dev)] = dmu  # the multipliers of the other shards' rows do not enter this shard's outputs
        wg = torch.empty(whole.n_constraints, dtype=torch.float64, device=dev)
        wj = torch.empty(whole.nnz_jacobian, dtype=torch.float64, device=dev)
        wh = torch.empty(whole.nnz_hessian, dtype=torch.float64, device=dev)
        wJ = torch.empty(1, dtype=torch.float64, device=dev)
        whole.eval_all_dev(wz.data_ptr(), sigma, wmu.data_ptr(), wJ.data_ptr(), 0, wg.data_ptr(), wj.data_ptr(), wh.data_ptr())
        whole.synchronize()
        shard_ok = bool(np.array_equal(wg.cpu().numpy()[rows], ref_out[0]) and np.array_equal(wj.cpu().numpy()[jpos], ref_out[1]) and
                        np.array_equal(wh.cpu().numpy()[hpos], ref_out[2]) and
                        abs(J_total - float(wJ.item())) <= 1e-12 * max(1.0, abs(float(wJ.item()))))
        whole.close()
        del wz, wmu, wg, wj, wh
    elif mode == "batch_split":
        one = dto.Evaluator(prob, device=local_rank)
        shard_ok = True
        for b in (0, batch_local - 1):
            zb = dZs[0][b * ev.n_vars:(b + 1) * ev.n_vars].contiguous()
            mb = dmu[b * ev.n_constraints:(b + 1) * ev.n_constraints].contiguous()
            og = torch.empty(ev.n_constraints, dtype=torch.float64, device=dev)
            oj = torch.empty(ev.nnz_jacobian, dtype=torch.float64, device=dev)
            oh = torch.empty(ev.nnz_hessian, dtype=torch.float64, device=dev)
            one.eval_all_dev(zb.data_ptr(), sigma, mb.data_ptr(), 0, 0, og.data_ptr(), oj.data_ptr(), oh.data_ptr())
            one.synchronize()
            shard_ok = shard_ok and bool(np.array_equal(og.cpu().numpy(), ref_out[0][b * ev.n_constraints:(b + 1) * ev.n_constraints]) and
                                         np.array_equal(oj.cpu().numpy(), ref_out[1][b * ev.nnz_jacobian:(b + 1) * ev.nnz_jacobian]) and
                                         np.array_equal(oh.cpu().numpy(), ref_out[2][b * ev.nnz_hessian:(b + 1) * ev.nnz_hessian]))
        one.close()

    if args.no_e2e:
        if rank == 0:
            print(json.dumps({"workload": workload, "ms_per_step": dev_ms / steps, "kernel_ms": k1_ms / max(k1_n, 1), "gpu_launches": int(launches),
                              "note": "--no-e2e: device-resident loop only"}), flush=True)
        ev.close()
        return None
    # ---- end-to-end through the host-pointer C ABI ------------------------------------------------
    # Host buffers as a solver holds them: page-locked Z / mu inputs, its own Jacobian / Hessian value arrays registered
    # once with the handle (dto_register_outputs: structural constants written once, value-dependent entries per call).
    # Every timed step is a NEW iterate (three iterates in rotation), so the upload of Z and mu is part of every step.
    n_iter = 3
    e2e_steps, e2e_warm = (steps, warmup) if full else (max(3, steps // 4), 2)
    hZs = [torch.from_numpy(Z + 1e-3 * i * rng.standard_normal(Z.size)).pin_memory() for i in range(n_iter)]
    hmus = [torch.from_numpy(rng.random(mu.size)).pin_memory() for _ in range(n_iter)]
    hZs[0].copy_(torch.from_numpy(Z))
    hmus[0].copy_(torch.from_numpy(mu))
    hJ = torch.empty(batch_local, dtype=torch.float64).pin_memory()
    hgrad = torch.empty(n_grad, dtype=torch.float64).pin_memory()
    hg = torch.empty(batch_local * ev.n_constraints, dtype=torch.float64).pin_memory()
    hjac = torch.empty(batch_local * ev.nnz_jacobian, dtype=torch.float64).pin_memory()
    hhess = torch.empty(batch_local * ev.nnz_hessian, dtype=torch.float64).pin_memory()
    nzs, nmus = [a.numpy() for a in hZs], [a.numpy() for a in hmus]
    outs = [a.numpy() for a in (hJ, hgrad, hg, hjac, hhess)]
    registered = False
    if batch_local == 1 and not args.no_register:
        ev.register_outputs(outs[3], outs[4])
        registered = True

    def step_fused(i):
        ev.eval_all(nzs[i % n_iter], sigma, nmus[i % n_iter], *outs)  # synchronises the stream before returning

    def step_sequence(i):
        # the five MOI callbacks as Ipopt / MadNLP issue them on one iterate (src/solvers/ipopt_solver/solver.jl:85)
        zi, mi = nzs[i % n_iter], nmus[i % n_iter]
        if linked:
            ev.upload(zi)  # linked shards: every rank uploads every iterate once (pushes the halo knot)
        outs[0][:] = ev.eval_objective(zi)
        ev.eval_objective_gradient(outs[1], zi)
        ev.eval_constraint(outs[2], zi)
        ev.eval_constraint_jacobian(outs[3], zi)
        ev.eval_hessian_lagrangian(outs[4], zi, sigma, mi)

    def time_host(step):
        for i in range(e2e_warm):
            step(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            step(i)
        barrier()
        return time.perf_counter() - t0

    e2e_fused_s = d2h_fused = None
    if full and not linked:
        e2e_fused_s = time_host(step_fused)
        d2h_fused = ev.last_d2h_bytes  # what crossed PCIe in the last fused call
    l_seq0 = ev.launch_count
    e2e_seq_s = time_host(step_sequence)
    seq_launches = (ev.launch_count - l_seq0) / (e2e_steps + e2e_warm)
    # bytes of one sequence step: measured callback by callback on one more new iterate
    zi = nzs[0] + 1e-6
    d2h_seq = 0
    if linked:
        ev.upload(zi)
    ev.eval_objective(zi)
    d2h_seq += ev.last_d2h_bytes
    ev.eval_objective_gradient(outs[1], zi)
    d2h_seq += ev.last_d2h_bytes
    ev.eval_constraint(outs[2], zi)
    d2h_seq += ev.last_d2h_bytes  # with registered outputs this includes the Jacobian that leaves on the side
    ev.eval_constraint_jacobian(outs[3], zi)
    d2h_seq += ev.last_d2h_bytes
    ev.eval_hessian_lagrangian(outs[4], zi, sigma, nmus[0])
    d2h_seq += ev.last_d2h_bytes
    h2d = 8 * (Z.size + mu.size)
    d2h_outputs = 8 * (hJ.numel() + hgrad.numel() + hg.numel() + hjac.numel() + hhess.numel())

    # parity guard on the timed outputs: the device-resident and host paths (callback sequence and fused) must agree bit for bit
    step_sequence(0)
    same_seq = bool(np.array_equal(outs[3], ref_out[1]) and np.array_equal(outs[4], ref_out[2]) and np.array_equal(outs[2], ref_out[0]))
    same = None
    if full and not linked:
        step_fused(0)
        same = bool(np.array_equal(outs[3], ref_out[1]) and np.array_equal(outs[4], ref_out[2]))
    if registered:
        ev.unregister_outputs()

    # ---- max over ranks ---------------------------------------------------------------------------
    agg = torch.tensor([dev_ms, e2e_seq_s, k1_ms / max(k1_n, 1), e2e_fused_s or 0.0, 0.0 if shard_ok in (None, True) else 1.0, 0.0 if same_seq else 1.0],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_s_max, k1_avg_ms, e2e_fused_s_max, shard_bad, seq_bad = agg.tolist()

    line = None
    if rank == 0:
        # units: problem evaluations.  replicas: one problem per rank per step (weak); knot_shards: the ranks
        # share ONE problem (strong); batch_split: the ranks share the batch (strong)
        per_step = {"replicas": world, "knot_shards": 1, "batch_split": WORKLOADS[workload].get("batch", 1)}[mode]
        value = per_step * steps / (dev_ms_max * 1e-3)
        e2e_value = per_step * e2e_steps / e2e_s_max
        # algorithmic flops of ONE launch of the dominant kernel on this rank
        n_interval_kernels = max(1, sum(1 for i in prob.integrators if type(i).__name__ != "DerivativeIntegrator"))
        intervals_per_launch = {"replicas": t.N - 1, "knot_shards": int(ev.n_dynamics_constraints // max(1, sum(i.x_dim for i in prob.integrators))),
                                "batch_split": batch_local * (t.N - 1)}[mode]
        tdb = type(prob.integrators[0]).__name__ == "TimeDependentBilinearIntegrator"
        rhs_avg = tdb_rhs_per_interval(prob, Z) if tdb else None  # what the kernels execute at this iterate (columns sized per interval)
        per_interval = canonical_flops_per_tdb_interval(n, m, prob.integrators[0].spline_order, rhs=rhs_avg) if tdb else canonical_flops_per_interval(n, m)
        flops_launch = per_interval * intervals_per_launch
        achieved = flops_launch / (k1_avg_ms * 1e-3) * 1e-12
        traffic, traffic_src = recorded_traffic(workload, ev.kernel_variant(0)) if world == 1 or mode == "replicas" else (None, None)
        out_bytes_dev = 8 * (2 * Z.size + 2 * mu.size + batch_local * (ev.n_constraints + ev.nnz_jacobian + ev.nnz_hessian))
        line = {
            "metric": "full NLP evals/sec (constraint+Jacobian+Hessian)", "value": value, "unit": "evals/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": dev_ms_max / steps, "higher_is_better": True,
            "scaling": "weak" if mode == "replicas" else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(workload_config(workload, prob, mode),
                           l2="256 MB memset between timed steps (outside the per-step CUDA events)",
                           outputs="value: outputs left in HBM (dto_eval_all_dev); e2e: the five callbacks (and, beside it, the fused dto_eval_all) with "
                                   "page-locked host buffers; the Jacobian / Hessian value arrays are registered with the handle once "
                                   "(dto_register_outputs: structural constants written once, only value-dependent entries cross PCIe per call; "
                                   "--no-register: plain buffers, host threads write the Hessian's structural zeros); knot-range pipeline: D2H of "
                                   "finished ranges overlaps the next range",
                           kernel_variant=ev.kernel_variant(0)),
            # headline e2e: the call sequence a solver makes (five separate C-ABI callbacks per iterate); the fused
            # single call (dto_eval_all, what benchmark/benchmarks.jl's loop amounts to) beside it
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_seq,
                    "ms_per_step": e2e_s_max / e2e_steps * 1e3, "matches_device_path": seq_bad == 0.0, "output_bytes_per_step": d2h_outputs,
                    "call": "dto_eval_objective + dto_eval_gradient + dto_eval_constraint + dto_eval_jacobian + dto_eval_hessian on a new iterate every step",
                    "outputs_registered": registered, "gpu_launches_per_step": seq_launches, "steps": e2e_steps},
            "gpu_launches": int(launches),
            "roofline": {
                "bound": "tensor", "achieved": achieved, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / FP64_PEAK_TFLOPS,
                "traffic": traffic, "traffic_unit": "bytes per launch (dram read + write, ncu --set full)", "traffic_source": traffic_src,
                "kernel": "time-dependent bilinear interval kernels (K7: tdb_dmma_kernel + tdb_exp_kernel)" if tdb else "bilinear interval kernel (K1)",
                "kernel_ms": k1_avg_ms,
                "kernel_share_of_step": k1_avg_ms * n_interval_kernels / (dev_ms_max / steps),
                "algorithmic_flops_per_launch": flops_launch,
                "peak_source": "FP64 DMMA m8n8k4 saturation measured on this pool (profiles/r01_fp64_peaks_and_box_probe.log); "
                               "MEASURED_PEAKS.json carries no FP64 figure; cuBLAS DGEMM 8192^3 measured 35.5 TFLOP/s",
                "hbm_gbs_step": out_bytes_dev / (dev_ms_max / steps * 1e-3) * 1e-9,
            },
        }
        if tdb:
            line["roofline"]["rhs_per_interval"] = rhs_avg
            line["roofline"]["rhs_note"] = ("right-hand sides executed per interval (extrapolation columns sized per interval from the iterate; 80 with "
                                            "eight columns everywhere, DTO_B200_TDB_TOL=0): the flop count is per executed right-hand side")
        if e2e_fused_s is not None:
            line["e2e"]["fused"] = {"call": "dto_eval_all", "value": per_step * e2e_steps / e2e_fused_s_max, "ms_per_step": e2e_fused_s_max / e2e_steps * 1e3,
                                    "d2h_bytes_per_step": d2h_fused, "matches_device_path": same}
            line["e2e"]["sequence_over_fused"] = e2e_s_max / e2e_fused_s_max
        if shard_ok is not None:
            line["shard_matches_single_gpu"] = shard_bad == 0.0
        if linked:
            line["scalar_reduce"] = "violation + exchange windows over NVLink peer memory in one kernel (dto_shard_scalars_dev)" if args.scalar_reduce == "peer" else "NCCL all_reduce x2"
        if full:
            line["clocks"] = sampler.summary()
            line["wall_s_timed_region"] = t_wall
            if not args.no_cpu_baseline and world == 1 and not tdb:  # the CPU baseline is timed on rank 0 of the single-GPU run only
                try:
                    threads = os.cpu_count() or 1
                    rate, info = cpu_port_rate(prob, args.cpu_sample, threads)
                    line["cpu_baseline"] = {"value": rate, "unit": "evals/s", "cores": info["threads"], "kind": "port", "sample": info["sample"]}
                    # the stronger CPU baseline: the same jets over the ACTIVE directions only (x, u, dt) instead of all 2z
                    rate2, info2 = cpu_port_rate(prob, 4 * args.cpu_sample, threads, all_dirs=False)
                    line["cpu_baseline_active_dirs"] = {"value": rate2, "unit": "evals/s", "cores": info2["threads"], "kind": "port", "sample": info2["sample"]}
                except Exception as e:  # the baseline must never take the GPU number down with it
                    line["cpu_baseline"] = {"value": None, "unit": "evals/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    del dZs, dmu, dg, djac, dhess, flush, hjac, hhess
    ev.close()
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "c2", "c3", "c4", "c5"],
                    help="all (default): the c2 headline line with short c3/c4/c5 runs embedded under `extra`")
    ap.add_argument("--cpu-sample", type=int, default=256, help="knot intervals timed for cpu_baseline (about 30 CPU-seconds at c2)")
    ap.add_argument("--ref-sample", type=int, default=64, help="knot intervals per step of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-register", action="store_true", help="e2e with plain (unregistered) output buffers")
    ap.add_argument("--no-extra", action="store_true", help="skip the embedded c3/c4/c5 runs of the default workload")
    ap.add_argument("--no-e2e", action="store_true", help="device-resident loop only (profiling: the ncu launch list of one step)")
    ap.add_argument("--scalar-reduce", default="peer", choices=["peer", "nccl"], help="knot shards: objective/violation reduction")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the headline workload (rank 0: objective, gradient, constraint, "
                         "jacobian, hessian values) as DIR/<name>.npy, float64; arrays above 2^20 entries as a fixed seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA evaluator (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    # host threads of the handle (they write the Hessian's structural zeros into UNREGISTERED buffers on the host-pointer
    # path): share the box's cores between the ranks, never fewer than 3 (below that the library delivers whole arrays)
    os.environ.setdefault("DTO_B200_HOST_THREADS", str(max(3, min(4, (os.cpu_count() or 4) // (2 * world)))))

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the evaluator has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    kw = dict(rank=rank, world=world, local_rank=local_rank)
    if args.workload != "all":
        line = run_workload(args, args.workload, args.steps, args.warmup, full=True, **kw)
    else:
        extra = {}
        if not args.no_extra:
            for w in ("c3", "c4", "c5"):
                try:
                    ln = run_workload(args, w, max(5, args.steps // 5), 3, full=False, **kw)
                except Exception as e:  # an extra must never take the headline down with it
                    if world > 1:
                        raise
                    ln = {"error": f"{type(e).__name__}: {e}"}
                if rank == 0:
                    extra[w] = {k: ln[k] for k in ("value", "unit", "ms_per_step", "scaling", "steps", "config", "e2e", "roofline", "gpu_launches",
                                                   "shard_matches_single_gpu", "scalar_reduce", "error") if k in ln}
                    if "config" in extra[w]:
                        extra[w]["config"] = {k: ln["config"][k] for k in ("workload", "per_rank", "kernel_variant")}
        line = run_workload(args, "c2", args.steps, args.warmup, full=True, **kw)
        if rank == 0 and extra:
            line["extra"] = extra
    if rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
