"""Time the per-sample fused energy (reduction="none") against the "mean" launch and against one launch per sample.

    python tools/bench_per_sample.py [--out profiles/r5_per_sample.jsonl] [--K 50] [--reps 5]

At 256^2 x 64, 512^2 x 16 and 64^3 x 16 (the bench.py batch shapes; u, nu, f and two Dirichlet masks):
  energy_mean            one fused launch, reduction="mean" (loss + grad_u)
  energy_none            one fused launch, reduction="none" ((B,) loss + grad_u)
  energy_B_launches      B launches of one sample each (what per-sample values cost without "none"); us per batch
  bwd_scalar_cotangent   the backward's gradient scaling with a 0-dim grad_output != 1 (dn_scale_inplace_f32)
  bwd_sample_cotangent   the same with a (B,) grad_output (dn_scale_per_sample_f32)
K steps are captured in one CUDA graph and replayed; every case rotates over enough input sets that the bytes it moves
per rotation exceed 400 MB (well beyond the 126 MB L2); CUDA events; median of `reps` replays.  One JSON line per
(workload, case) with the device name and power limit; `none_over_mean` compares the two fused launches.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_input_grads import ROTATE_BYTES, device_info, timed  # noqa: E402
from diffnet_b200 import ops  # noqa: E402

WORKLOADS = [((256, 256), 64), ((512, 512), 16), ((64, 64, 64), 16)]


def geometry(sp):
    h = 1.0 / (sp[-1] - 1)
    if len(sp) == 2:
        return ops.Geometry(2, sp[1], sp[0], 1, h, h, 0.0, 2)
    return ops.Geometry(3, sp[2], sp[1], sp[0], h, h, h, 2)


def run(args):
    if not torch.cuda.is_available():
        raise SystemExit("bench_per_sample.py times the B200 kernels: no CUDA device")
    name, power = device_info()
    rows = []
    for sp, B in WORKLOADS:
        geom = geometry(sp)
        dof = B
        for s in sp:
            dof *= s
        nbytes = 24 * dof                                 # u, nu, f, 2 masks read; grad_u written
        nsets = max(2, -(-ROTATE_BYTES // nbytes))
        g = torch.Generator(device="cuda").manual_seed(0)
        sets = []
        for _ in range(nsets):
            shp = (B,) + sp
            m0 = torch.zeros(shp, device="cuda"); m0[..., 0] = 1
            m1 = torch.zeros(shp, device="cuda"); m1[..., -1] = 1
            sets.append(dict(u=torch.randn(shp, generator=g, device="cuda"),
                             nu=torch.rand(shp, generator=g, device="cuda") + 0.5,
                             f=torch.randn(shp, generator=g, device="cuda"), d=[(m0, 1.0), (m1, 0.0)],
                             grad=torch.randn(shp, generator=g, device="cuda")))
        half = torch.tensor(0.5, device="cuda")
        w = torch.rand(B, generator=g, device="cuda") + 0.5

        def energy(i, reduction):
            s = sets[i]
            return ops.energy_raw(geom, s["u"], nu=s["nu"], f=s["f"], dirichlet=s["d"], reduction=reduction)

        def one_by_one(i):
            s = sets[i]
            for b in range(B):
                ops.energy_raw(geom, s["u"][b:b + 1], nu=s["nu"][b:b + 1], f=s["f"][b:b + 1],
                               dirichlet=[(m[b:b + 1], v) for m, v in s["d"]], reduction="sum")

        cases = {
            "energy_mean": (lambda i: energy(i, "mean"), nbytes, args.K),
            "energy_none": (lambda i: energy(i, "none"), nbytes, args.K),
            "energy_B_launches": (one_by_one, nbytes, max(2, args.K // B)),
            "bwd_scalar_cotangent": (lambda i: ops.scale_inplace_(sets[i]["grad"], half), 8 * dof, args.K),
            "bwd_sample_cotangent": (lambda i: ops.scale_per_sample_(sets[i]["grad"], w), 8 * dof, args.K),
        }
        us = {}
        for case, (step, nb, K) in cases.items():
            n = min(nsets, max(2, -(-ROTATE_BYTES // nb)))
            ms = timed(step, n, K, args.reps)
            us[case] = ms * 1e3
            row = dict(workload=f"{'x'.join(map(str, sp))}x{B}", case=case, us_per_step=round(ms * 1e3, 2),
                       algorithmic_MB=round(nb / 1e6, 1), GBps=round(nb / (ms * 1e-3) / 1e9, 1), device=name,
                       power_limit=power, K=K, reps=args.reps, input_sets=n)
            if case == "energy_none":
                row["none_over_mean"] = round(us["energy_none"] / us["energy_mean"], 4)
            if case == "energy_B_launches":
                row["over_none"] = round(us["energy_B_launches"] / us["energy_none"], 2)
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
    run(ap.parse_args())
