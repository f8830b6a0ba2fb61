"""Time the input-gradient launches (dn_fem_{energy,residual}_input_grads_*) the way bench.py times the fused loss.

    python tools/bench_input_grads.py [--out FILE.jsonl] [--K 50] [--reps 5]

K launches are captured in one CUDA graph and replayed; each case rotates over enough input sets that the bytes it moves
per rotation exceed 400 MB (every launch streams from HBM, not from the 126 MB L2); CUDA events; median of `reps`
replays.  The peak is the measured copy peak bench.py's roofline uses (bench.measured_peak_gbs).  Bytes are
algorithmic: every field the launch reads and every output it writes, computed from the shapes.  One JSON line per (workload, launch), with the device name and
power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import measured_peak_gbs  # noqa: E402
from diffnet_b200 import ops  # noqa: E402

ROTATE_BYTES = 400_000_000     # as bench.copy_reference: well beyond the 126 MB L2


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception:   # noqa: BLE001
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def timed(step, nsets, K, reps):
    """ms per launch: K launches (rotating over nsets input sets) replayed from one CUDA graph, median of reps."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(nsets):                  # warm every set (module load, workspace)
            step(i)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for i in range(K):
            step(i % nsets)
    graph.replay()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) / K)
    return sorted(times)[len(times) // 2]




def workload(nsd):
    if nsd == 2:
        B, sp, h = 64, (256, 256), 1.0 / 255
        geom = ops.Geometry(2, 256, 256, 1, h, h, 0.0, 2)
    else:
        B, sp, h = 16, (64, 64, 64), 1.0 / 63
        geom = ops.Geometry(3, 64, 64, 64, h, h, h, 2)
    return B, sp, geom


def run(args):
    name, power = device_info()
    peak, peak_src = measured_peak_gbs()
    rows = []
    for nsd in (2, 3):
        B, sp, geom = workload(nsd)
        dof = B
        for s in sp:
            dof *= s
        ngp = geom.ngp_1d ** nsd
        nel = B
        for s in sp:
            nel *= s - 1
        # every case rotates over enough sets that the bytes IT moves per rotation exceed ROTATE_BYTES (> 3x the L2)
        nsets = max(2, -(-ROTATE_BYTES // (16 * dof)))          # the smallest case (energy_df) needs the most sets
        g = torch.Generator(device="cuda").manual_seed(0)
        sets = []
        for _ in range(nsets):
            shp = (B,) + sp
            m0 = torch.zeros(shp, device="cuda"); m0[..., 0] = 1
            m1 = torch.zeros(shp, device="cuda"); m1[..., -1] = 1
            sets.append(dict(u=torch.randn(shp, generator=g, device="cuda"),
                             nu=torch.rand(shp, generator=g, device="cuda") + 0.5,
                             f=torch.randn(shp, generator=g, device="cuda"),
                             R=torch.randn(shp, generator=g, device="cuda"),
                             m0=m0, m1=m1, blob=(torch.rand(shp, generator=g, device="cuda") > 0.8).float(),
                             v=torch.randn(shp, generator=g, device="cuda"),
                             fgp=torch.randn((B, ngp) + tuple(s - 1 for s in sp), generator=g, device="cuda")))
        two = lambda s: [(s["m0"], 1.0), (s["m1"], 0.0)]   # noqa: E731
        cases = {
            "energy_df": (lambda i: ops.energy_input_grads_raw(geom, sets[i]["u"], f=sets[i]["f"],
                                                               dirichlet=two(sets[i]), want_f=True),
                          16 * dof),                     # u, 2 masks -> grad_f
            "energy_dfgp": (lambda i: ops.energy_input_grads_raw(geom, sets[i]["u"], f_gp=sets[i]["fgp"],
                                                                 dirichlet=two(sets[i]), want_f_gp=True),
                            12 * dof + 4 * ngp * nel),   # u, 2 masks -> grad_f_gp
            "energy_dubc": (lambda i: ops.energy_input_grads_raw(geom, sets[i]["u"], nu=sets[i]["nu"], f=sets[i]["f"],
                                                                 dirichlet=[(sets[i]["blob"], sets[i]["v"])],
                                                                 want_values=(True,)),
                            24 * dof),                   # u, nu, f, mask, value field -> grad value
            "residual_dnu_df": (lambda i: ops.residual_input_grads_raw(geom, sets[i]["u"], sets[i]["R"], nu=sets[i]["nu"],
                                                                       f=sets[i]["f"], dirichlet=two(sets[i]),
                                                                       want_nu=True, want_f=True),
                                24 * dof),               # u, R, 2 masks -> grad_nu, grad_f (nu, f: not read)
            "fused_forward": (lambda i: ops.energy_raw(geom, sets[i]["u"], nu=sets[i]["nu"], f=sets[i]["f"],
                                                       dirichlet=two(sets[i])),
                              24 * dof),                 # u, nu, f, 2 masks -> grad_u
            "fused_forward_plus_df": (lambda i: (ops.energy_raw(geom, sets[i]["u"], nu=sets[i]["nu"], f=sets[i]["f"],
                                                                dirichlet=two(sets[i])),
                                                 ops.energy_input_grads_raw(geom, sets[i]["u"], f=sets[i]["f"],
                                                                            dirichlet=two(sets[i]), want_f=True)),
                                      40 * dof),
        }
        for case, (step, nbytes) in cases.items():
            n = min(nsets, max(2, -(-ROTATE_BYTES // nbytes)))
            ms = timed(step, n, args.K, args.reps)
            gbs = nbytes / (ms * 1e-3) / 1e9
            row = dict(workload=f"{'x'.join(map(str, sp))}x{B}", launch=case, us_per_launch=round(ms * 1e3, 2),
                       algorithmic_MB=round(nbytes / 1e6, 1), GBps=round(gbs, 1), copy_peak_GBps=round(peak, 1),
                       frac_of_copy_peak=round(gbs / peak, 3), peak_source=peak_src, device=name, power_limit=power, K=args.K,
                       reps=args.reps, input_sets=n)
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for r in rows:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--K", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_input_grads: needs a CUDA device (no CPU timing)")
    run(a)
