"""What a knot program costs against the catalogue entry it replaces, on the c2 shape (quantum_gate_problem: 16 levels,
n = 32, 4 drives, N = 2000) plus two terms: a TerminalObjective iso-infidelity and norm(u) <= 1 at every knot.

Variants, built from the same seeded problem:
  catalogue   IsoInfidelity + NormMinus (device catalogue)
  program     the same two functions written as KnotPrograms
  program100  `program` plus a 100-operation, 32-variable program constraint on x at every knot

Timing: dto_eval_all_dev (sigma = 1, every output) with CUDA events around each step, L2 flushed between steps as in
bench.py, variants alternated in blocks within one process after a warm-up.  --profile instead records per-kernel
device time with torch.profiler (a separate run: tracing slows the host).  Also checks that catalogue and program
outputs agree (relative to each output's max-norm) and prints the GPU name and power limit.

  python tools/knot_program_timing.py [--steps 240] [--block 20] [--profile] [--out FILE.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import dto_b200 as dto  # noqa: E402
from dto_b200 import problem_templates as pt  # noqa: E402


def wide_program(nv=32):
    """a 100-operation function of 32 variables"""
    return dto.KnotProgram(lambda v: [sum(np.tanh(v[i]) * v[(i + 5) % nv] for i in range(22)) - 0.5])


def problems(N):
    base = pt.quantum_gate_problem(N=N, levels=16, n_drives=4)
    traj = base.trajectory
    n = traj.dims["x"]
    h = n // 2
    goal = np.zeros(n)
    goal[1] = 1.0

    def build(infid, unorm, extra=None):
        J = base.objective + dto.TerminalObjective(infid, "x", traj, Q=1.0)
        cons = [dto.NonlinearKnotPointConstraint(unorm, "u", traj, equality=False)]
        if extra is not None:
            cons.append(dto.NonlinearKnotPointConstraint(extra, "x", traj, equality=False))
        return dto.DirectTrajOptProblem(traj, J, base.integrators, constraints=cons)

    infid = dto.KnotProgram(lambda v, p: 1.0 - ((v[:h] @ p[:h] + v[h:] @ p[h:]) ** 2 + (v[h:] @ p[:h] - v[:h] @ p[h:]) ** 2), params=goal)
    unorm = dto.KnotProgram(lambda v: [np.sqrt(v @ v) - 1.0])
    return {
        "catalogue": build(dto.IsoInfidelity(goal), dto.NormMinus(1.0)),
        "program": build(infid, unorm),
        "program100": build(infid, unorm, wide_program()),
    }


def gpu_info():
    import torch

    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip()
    except Exception as e:  # the measurement stands without it, but says so
        smi = f"nvidia-smi unavailable: {e}"
    return {"torch_name": name, "nvidia_smi": smi}


class Runner:
    def __init__(self, prob, rng_seed=0):
        import torch

        self.ev = ev = dto.Evaluator(prob)
        rng = np.random.default_rng(rng_seed)
        Z = prob.trajectory.vec()
        Z = Z + 0.01 * rng.standard_normal(Z.size)
        mu = rng.random(ev.n_constraints)
        dev = torch.device("cuda")
        f64 = dict(dtype=torch.float64, device=dev)
        self.Z, self.mu = torch.tensor(Z, **f64), torch.tensor(mu, **f64)
        self.J = torch.empty(1, **f64)
        self.grad = torch.empty(ev.n_vars, **f64)
        self.g = torch.empty(ev.n_constraints, **f64)
        self.jac = torch.empty(ev.nnz_jacobian, **f64)
        self.hess = torch.empty(ev.nnz_hessian, **f64)
        self.stream = torch.cuda.ExternalStream(ev.stream)

    def step(self):
        self.ev.eval_all_dev(self.Z.data_ptr(), 1.0, self.mu.data_ptr(), self.J.data_ptr(), self.grad.data_ptr(), self.g.data_ptr(),
                             self.jac.data_ptr(), self.hess.data_ptr())

    def outputs(self):
        import torch

        torch.cuda.synchronize()
        return {k: getattr(self, k).cpu().numpy() for k in ("J", "grad", "g", "jac", "hess")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=240, help="timed steps per variant")
    ap.add_argument("--block", type=int, default=20, help="steps per variant before switching to the next")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", help="also write the result as JSON to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("knot_program_timing: no CUDA device (there is no CPU timing of this path)")
    info = gpu_info()
    print(json.dumps(info))
    probs = problems(args.N)
    runners = {k: Runner(p) for k, p in probs.items()}
    for k, r in runners.items():
        c = r.ev.prob.nonlinear_constraints()
        print(f"{k}: n_cons {r.ev.n_constraints}, nnz_jac {r.ev.nnz_jacobian}, nnz_hess {r.ev.nnz_hessian}, "
              f"program ops {[int(x.g.trace(x.var_dim).ops.shape[0]) for x in c if isinstance(x.g, dto.KnotProgram)]}")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")  # > 126 MB L2
    for r in runners.values():
        with torch.cuda.stream(r.stream):
            for _ in range(args.warmup):
                r.step()
    torch.cuda.synchronize()

    # agreement of the catalogue and program forms (same problem, same iterate)
    ref, got = runners["catalogue"].outputs(), runners["program"].outputs()
    agree = {k: float(np.abs(got[k] - ref[k]).max() / max(np.abs(ref[k]).max(), 1e-300)) for k in ref}
    print("catalogue vs program, max relative difference:", json.dumps(agree))
    result = {"gpu": info, "N": args.N, "agreement_rel": agree, "agree_1e-13": all(v <= 1e-13 for v in agree.values())}

    if args.profile:
        from torch.profiler import ProfilerActivity, profile

        per = {}
        for k, r in runners.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                with torch.cuda.stream(r.stream):
                    for _ in range(args.block):
                        r.step()
                torch.cuda.synchronize()
            tab = {}
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                if t > 0:
                    tab[e.key] = {"us_per_step": t / args.block, "calls_per_step": e.count / args.block}
            per[k] = dict(sorted(tab.items(), key=lambda kv: -kv[1]["us_per_step"]))
            print(f"--- {k}: per-kernel device time (us / step)")
            for name, v in list(per[k].items())[:12]:
                print(f"  {v['us_per_step']:10.1f}  x{v['calls_per_step']:.0f}  {name[:110]}")
        result["profile"] = per
    else:
        times = {k: [] for k in runners}
        reps = max(1, args.steps // args.block)
        for _ in range(reps):
            for k, r in runners.items():
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.block)]
                with torch.cuda.stream(r.stream):
                    for e0, e1 in evs:
                        flush.zero_()
                        e0.record(r.stream)
                        r.step()
                        e1.record(r.stream)
                torch.cuda.synchronize()
                times[k] += [e0.elapsed_time(e1) for e0, e1 in evs]
        stats = {k: {"steps": len(v), "median_ms": float(np.median(v)), "p10_ms": float(np.percentile(v, 10)),
                     "p90_ms": float(np.percentile(v, 90))} for k, v in times.items()}
        base = stats["catalogue"]["median_ms"]
        for k, s in stats.items():
            s["vs_catalogue"] = s["median_ms"] / base
            print(f"{k:11s} median {s['median_ms']:.4f} ms (p10 {s['p10_ms']:.4f}, p90 {s['p90_ms']:.4f}) over {s['steps']} steps, "
                  f"x{s['vs_catalogue']:.3f} of catalogue")
        result["timing"] = stats
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    for r in runners.values():
        r.ev.close()


if __name__ == "__main__":
    main()
