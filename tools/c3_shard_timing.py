"""Config c3 (time-dependent bilinear, linear spline, n = 64, 2 drives, N = 1000) in knot-range shards: what the boundary
Hessian block exchange buys.  Device-resident steps (upload_dev of a new iterate + eval_all_dev with the Hessian), one JSON
line per measurement.

  one GPU   for world = 1, 2, 4, 8 the knot_ranges(N, world) shards live on cuda:0, linked with dto_shard_link_local.  Every
            step uploads a new iterate on every shard (rank order), then each shard's evaluation is timed ALONE (CUDA
            events on its stream, synchronised before the next shard starts), in rank order, so each wait for a
            neighbour is already satisfied: the per-rank step time of a one-GPU-per-rank run (the proxy of
            tools/c4_size_sweep.py).  speedup = t(1) / max over shares.  A profiled pass gives the device time of the
            block push and receive kernels per step.
  several   (torch.cuda.device_count() > 1): one shard per device in this process, linked locally, every shard's step
            enqueued before any synchronises; per-rank event times, their max and the efficiency t(1) / (world * max).

usage: python tools/c3_shard_timing.py [--steps 20] [--warmup 3] [--out FILE]   (one JSON line per measurement)"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import dto_b200 as dto
from dto_b200 import problem_templates as pt
from dto_b200.sharding import knot_ranges

N, N_STATE, N_DRIVES = 1000, 64, 2


def box():
    name = torch.cuda.get_device_name(0)
    try:  # read-only query
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        lim = r.stdout.strip()
    except Exception:
        lim = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": lim, "date": time.strftime("%Y-%m-%d")}


class Shard:
    """one linked shard with two device-resident iterates in rotation and its device outputs"""

    def __init__(self, prob, cut, device, rng):
        self.dev = torch.device("cuda", device)
        self.ev = dto.Evaluator(prob, shard=cut, device=device)
        L = self.ev.shard_layout
        Z0 = prob.trajectory.vec()
        self.Z = [torch.from_numpy(Z0[L.z_begin:L.z_halo_end] + 0.01 * rng.standard_normal(L.z_halo_end - L.z_begin)).to(self.dev)
                  for _ in range(2)]
        for z in self.Z:
            if L.z_halo_end > L.z_end:
                z[L.z_end - L.z_begin:] = float("nan")  # linked: the halo knot comes through the window
        ev = self.ev
        self.mu = torch.rand(max(ev.n_constraints, 1), dtype=torch.float64, device=self.dev)
        self.out = [torch.empty(max(k, 1), dtype=torch.float64, device=self.dev)
                    for k in (1, L.z_end - L.z_begin, ev.n_constraints, ev.nnz_jacobian, ev.nnz_hessian)]
        self.stream = torch.cuda.ExternalStream(ev.stream, device=self.dev)

    def upload(self, it):
        self.ev.upload_dev(self.Z[it & 1].data_ptr())

    def evaluate(self):
        self.ev.eval_all_dev(self.ev.local_Z_ptr, 1.0, self.mu.data_ptr(), *[o.data_ptr() for o in self.out])

    def timed(self, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.device(self.dev):
            e0.record(self.stream)
            fn()
            e1.record(self.stream)
        return e0, e1


def make(world, devices, seed=0):
    prob = pt.carrier_problem(N=N, state_dim=N_STATE, n_drives=N_DRIVES, spline_order=1)
    rng = np.random.default_rng(seed)
    shards = [Shard(prob, c, devices[r], rng) for r, c in enumerate(knot_ranges(N, world))]
    dto.Evaluator.shard_link_local([s.ev for s in shards])
    return shards


def one_gpu(world, steps, warmup):
    """per-share step time on cuda:0, shares stepped alone in rank order"""
    shards = make(world, [0] * world)
    up = [[] for _ in shards]
    ev_ms = [[] for _ in shards]
    for it in range(warmup + steps):
        for r, s in enumerate(shards):  # phase 1: every shard uploads the new iterate (pushes its first knot)
            e = s.timed(lambda: s.upload(it))
            s.ev.synchronize()
            if it >= warmup:
                up[r].append(e[0].elapsed_time(e[1]))
        for r, s in enumerate(shards):  # phase 2: each evaluation alone
            e = s.timed(s.evaluate)
            s.ev.synchronize()
            if it >= warmup:
                ev_ms[r].append(e[0].elapsed_time(e[1]))
    share = [float(np.median(a)) + float(np.median(b)) for a, b in zip(up, ev_ms)]
    # device time of the block exchange kernels per step (a profiled pass of its own)
    from torch.profiler import ProfilerActivity, profile

    prof_steps = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for it in range(prof_steps):
            for s in shards:
                s.upload(it)
                s.ev.synchronize()
            for s in shards:
                s.evaluate()
                s.ev.synchronize()
        torch.cuda.synchronize()
    push_us = recv_us = 0.0
    n_push = n_recv = 0
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            if "hs_push_kernel" in e.name:
                push_us += e.device_time
                n_push += 1
            elif "hs_receive_kernel" in e.name:
                recv_us += e.device_time
                n_recv += 1
    for s in shards:
        s.ev.close()
    return {"world": world, "share_ms": [round(x, 4) for x in share], "upload_ms": [round(float(np.median(a)), 4) for a in up],
            "eval_ms": [round(float(np.median(b)), 4) for b in ev_ms], "max_share_ms": round(max(share), 4),
            "push_kernel_us_per_launch": round(push_us / max(n_push, 1), 2), "receive_kernel_us_per_launch": round(recv_us / max(n_recv, 1), 2),
            "push_launches_per_step": n_push / prof_steps, "receive_launches_per_step": n_recv / prof_steps}


def several_gpus(world, steps, warmup):
    """one shard per device, every step enqueued on all shards before any synchronises"""
    shards = make(world, list(range(world)))
    per = [[] for _ in shards]
    wall = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        evs = []
        for s in shards:
            evs.append(s.timed(lambda: (s.upload(it), s.evaluate())))
        for s in shards:
            s.ev.synchronize()
        if it >= warmup:
            wall.append((time.perf_counter() - t0) * 1e3)
            for r, e in enumerate(evs):
                per[r].append(e[0].elapsed_time(e[1]))
    med = [float(np.median(p)) for p in per]
    for s in shards:
        s.ev.close()
    return {"world": world, "rank_ms": [round(x, 4) for x in med], "max_rank_ms": round(max(med), 4), "host_wall_ms": round(float(np.median(wall)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("c3_shard_timing: needs a CUDA device")
    info = box()
    lines = []
    t1 = None
    for world in (1, 2, 4, 8):
        r = one_gpu(world, a.steps, a.warmup)
        t1 = r["max_share_ms"] if world == 1 else t1
        r.update(mode="one GPU, shares stepped alone (per-rank step proxy)", projected_speedup=round(t1 / r["max_share_ms"], 3), **info)
        lines.append(r)
        print(json.dumps(r), flush=True)
    ndev = torch.cuda.device_count()
    for world in (2, 4, 8):
        if world > ndev:
            break
        r = several_gpus(world, a.steps, a.warmup)
        r.update(mode="one shard per GPU, one process, all enqueued before any synchronise", speedup=round(t1 / r["max_rank_ms"], 3),
                 efficiency=round(t1 / (world * r["max_rank_ms"]), 3), **info)
        lines.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
