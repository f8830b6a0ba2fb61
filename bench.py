#!/usr/bin/env python
"""bench.py -- FEM loss+grad throughput of the fused sm_100a kernels (and the reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (fused Poisson energy loss + gradient w.r.t. u) over one
batch of synthetic input.  Default workload = BASELINE.json configs[1]: Poisson 2-D parametric,
256 x 256 Q1 mesh, batch 64 per GPU, KL log-diffusivity, inputs (u, nu, f, bc1, bc2) fp32.

Prints ONE JSON line (rank 0).  Keys follow the driver contract; see DESIGN.md section 8.
  value     GDOF/s, whole job, inputs resident in HBM, K launches timed by CUDA events
            (replayed from one CUDA graph so the 15-us kernels are not host-launch bound)
  e2e       same metric through the public module API with PINNED HOST buffers: H2D of the
            step's five fields + launch + D2H of the loss inside the timed region
  roofline  algorithmic bytes (24 B/DOF) / measured launch duration vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle (= reference conv path restated, torch CPU) on this box's host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nsd, size, batch per GPU, bytes/DOF fwd+bwd, description)
    "poisson2d_param_256_b64": (2, 256, 64, 24, "Poisson 2D parametric 256x256 Q1, KL log-diffusivity, batch 64/GPU"),
    "poisson2d_param_256_b16": (2, 256, 16, 24, "scaling probe: 256x256, batch 16"),
    "poisson2d_param_256_b256": (2, 256, 256, 24, "scaling probe: 256x256, batch 256"),
    "poisson2d_param_256_b1024": (2, 256, 1024, 24, "scaling probe: 256x256, batch 1024"),
    "poisson2d_512_b16": (2, 512, 16, 24, "Poisson 2D 512x512 Q1, batch 16/GPU (roofline point)"),
    "ibn2d_512_b16": (2, 512, 16, 24, "IBN 2D irregular-domain Poisson, synthetic immersed silhouettes, 512x512, batch 16/GPU (configs[4])"),
    "poisson2d_512_b1": (2, 512, 1, 24, "Poisson 2D 512x512, batch 1 (IBN 2D single image; latency probe)"),
    "poisson2d_64_b1": (2, 64, 1, 24, "Poisson 2D non-parametric 64x64 (configs[0])"),
    "poisson3d_param_64_b16": (3, 64, 16, 20, "Poisson 3D parametric 64^3 Q1 hex, batch 16/GPU (u, source, sink, f)"),
    "poisson3d_128_b1": (3, 128, 1, 24, "Poisson 3D 128^3, variable nu, f, two masks (roofline point)"),
    "poisson3d_256_b1": (3, 256, 1, 20, "Poisson 3D non-parametric 256^3 (u, nu, bc1, f)"),
    # forcing given AT the Gauss points (e8_2d_poisson_mms.py:154-175): streamed as an assembled load vector (4 B/node)
    "mms2d_fgp_256_b64": (2, 256, 64, 24, "Poisson 2D 256x256, batch 64/GPU, forcing at the Gauss points (u, nu, b(f_gp), bc1, bc2)"),
    "mms3d_fgp_64_b16": (3, 64, 16, 20, "Poisson 3D 64^3, batch 16/GPU, nu == 1, forcing at the Gauss points (u, b(f_gp), source, sink)"),
    # one 256^3 field split into z-slabs over the ranks (strong scaling; halo exchange + loss all-reduce)
    "poisson3d_256_slab": (3, 256, 1, 20, "Poisson 3D non-parametric 256^3, z-slabs over all ranks, 1-plane halo exchange"),
}
DEFAULT = "poisson2d_param_256_b64"


def measured_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the
    committed ncu capture of this workload (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(name)
    except Exception:   # noqa: BLE001
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:   # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:   # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:   # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_inputs(name, device, seed):
    import torch
    from diffnet_b200.synthetic import ibn2d_batch, poisson2d_parametric_batch, poisson3d_parametric_batch
    nsd, size, B, _, _ = WORKLOADS[name]
    if nsd == 2:
        gen = ibn2d_batch if name.startswith("ibn2d") else poisson2d_parametric_batch
        u, inputs, f = gen(B, size, device, seed)
        if name.startswith("mms"):
            g = torch.Generator(device="cpu").manual_seed(seed + 11)
            f_gp = torch.randn(B, 4, size - 1, size - 1, generator=g).to(device)
            return dict(u=u, nu=inputs[:, 0:1], f_gp=f_gp, dirichlet=[(inputs[:, 1:2], 1.0), (inputs[:, 2:3], 0.0)],
                        c_k=0.5, _fields=[u, inputs, f_gp])
        return dict(u=u, nu=inputs[:, 0:1], f=f, dirichlet=[(inputs[:, 1:2], 1.0), (inputs[:, 2:3], 0.0)],
                    _fields=[u, inputs, f])
    u, src, sink, f = poisson3d_parametric_batch(B, size, device, seed)
    if name.startswith("mms"):
        g = torch.Generator(device="cpu").manual_seed(seed + 11)
        f_gp = torch.randn(B, 8, size - 1, size - 1, size - 1, generator=g).to(device)
        return dict(u=u, f_gp=f_gp, dirichlet=[(sink, 0.0), (src, 1.0)], c_k=0.5, _fields=[u, src, sink, f_gp])
    if name == "poisson3d_param_64_b16":       # IBN_3D.py:114-136: nu == 1
        return dict(u=u, f=f, dirichlet=[(sink, 0.0), (src, 1.0)], _fields=[u, src, sink, f])
    g = torch.Generator(device="cpu").manual_seed(seed + 7)
    nu = torch.exp(0.5 * torch.randn(u.shape, generator=g)).to(device)
    if name == "poisson3d_256_b1":             # solve_in_object_3d.py:75-102
        return dict(u=u, nu=nu, f=f + 500.0, dirichlet=[(src, 0.0)], c_k=0.5, _fields=[u, nu, src, f])
    return dict(u=u, nu=nu, f=f, dirichlet=[(sink, 0.0), (src, 1.0)], _fields=[u, nu, src, sink, f])


def make_fem(name):
    from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM
    nsd, size, B, _, _ = WORKLOADS[name]
    return (DiffNet2DFEM if nsd == 2 else DiffNet3DFEM)(None, domain_size=size, batch_size=B)


def call_kwargs(d):
    return {k: v for k, v in d.items() if not k.startswith("_") and k != "u"}


def nsets_for(name):
    """Input sets a timed run rotates through so that every step streams from HBM, not from the 126 MB L2."""
    nsd, size, B, bpd, _ = WORKLOADS[name]
    return min(64, max(2, int(-(-400e6 // (B * size ** nsd * bpd)))))


def shared_config(name, world):
    """The `config` object of the JSON line: identical for --impl ours and --impl reference (the
    driver compares them); everything arm-specific lives under `run`."""
    nsd, size, B, bpd, desc = WORKLOADS[name]
    n = nsets_for(name)
    return {"workload": name, "desc": desc, "batch_per_gpu": B, "grid": [size] * nsd,
            "dof_per_step_per_gpu": B * size ** nsd, "fields": "u, nu, f, bc1, bc2 (fp32)" if bpd == 24 else "4 fp32 nodal fields",
            "bytes_per_dof": bpd,
            "l2": f"GPU arm: inputs rotated over {n} buffer sets ({n * B * size ** nsd * bpd / 1e6:.0f} MB "
                  + ("> 126 MB L2" if n * B * size ** nsd * bpd > 126e6 else "-- fits the L2: a launch-latency probe, not a bandwidth number")
                  + "); CPU arm: host memory",
            "parallelism": f"dp{world} (batch sharded over the ranks, no data-path collective)"}


FLOPS_PER_DOF = {2: 90.0, 3: 280.0}     # closed-form fp32 operations per DOF, fwd + adjoint (SURVEY.md 8d)


def time_workload(name, dev, seed, K, W, reps, world=1, barrier=None, use_graph=True, keep_last=False):
    """Device-timed fused loss+gradient launches of one workload on this rank: K launches replayed
    from one CUDA graph, CUDA events, median of `reps`.  Returns ms per step (this rank) and the mode;
    with `keep_last`, also `last`: host copies of (loss, grad) of the last timed step."""
    import torch
    fem = make_fem(name)
    nsets = nsets_for(name)
    sets = [make_inputs(name, dev, seed=seed + i) for i in range(nsets)]
    kws = [call_kwargs(s) for s in sets]

    def launch(i):
        s = sets[i % nsets]
        return fem.energy_loss_and_grad(s["u"], **kws[i % nsets])

    for i in range(max(W, 3)):
        launch(i)
    torch.cuda.synchronize()
    mode, graph = "cuda_graph", None
    if use_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(2):
                    launch(i)                      # allocate this stream's workspace before capture
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for i in range(K):
                    out = launch(i)                # outputs are recycled by the graph's pool; the last stays live
            graph.replay()                         # one untimed replay
            torch.cuda.synchronize()
        except Exception as e:   # noqa: BLE001
            graph, mode = None, f"eager (graph capture failed: {type(e).__name__})"
            torch.cuda.synchronize()
    else:
        mode = "eager"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        if barrier is not None:
            barrier()
        else:
            torch.cuda.synchronize()
        e0.record()
        if graph is not None:
            graph.replay()
        else:
            for i in range(K):
                out = launch(i)
        e1.record()
        if barrier is not None:
            barrier()
        else:
            torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms_step = sorted(times)[len(times) // 2] / K
    res = {"ms_step": ms_step, "mode": mode, "sets": sets, "fem": fem, "nsets": nsets}
    if keep_last:
        res["last"] = {"loss": out[0].detach().cpu(), "grad": out[1].detach().cpu()}
    return res


DUMP_BYTES = 60_000_000     # --dump-outputs writes at most this much array data (64 MB with headroom)


def dump_outputs(out_dir, arrays):
    """Write each tensor of `arrays` as out_dir/<name>.npy (float32 / float64).  When the total exceeds
    DUMP_BYTES, every array is cut to about the same fraction of its elements: every `stride`-th flat
    element from an offset drawn by a generator seeded with 0, so the same shapes always give the same
    sample, and no index array is built."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    frac = min(1.0, DUMP_BYTES / max(total, 1))
    written = {}
    for name, t in arrays.items():
        flat = t.detach().cpu().reshape(-1)
        if flat.dtype not in (torch.float32, torch.float64):
            flat = flat.float()
        stride = -(-flat.numel() // max(1, int(flat.numel() * frac)))      # ceil: never above the budget
        if stride > 1:
            g = torch.Generator(device="cpu").manual_seed(0)
            offset = int(torch.randint(stride, (1,), generator=g))
            arr = flat[offset::stride].numpy()
        else:
            arr = flat.numpy().reshape(tuple(t.shape))
        np.save(os.path.join(out_dir, name + ".npy"), arr)
        written[name] = {"shape": list(t.shape), "stored": int(arr.size), "dtype": str(arr.dtype)}
    return written


def copy_reference(dev, nbytes, K=50, reps=3):
    """What a plain device copy achieves at THIS launch size: `b.copy_(a)` moving `nbytes` in total
    (nbytes/2 read + nbytes/2 written -- the same definition as MEASURED_PEAKS.json's hbm_gbs, which is
    taken at 4 GiB per launch), K launches replayed from one CUDA graph over rotating buffers larger
    than the L2, CUDA events.  The fixed per-launch cost (launch, ramp-up, drain) that separates a
    100 MB launch from the multi-GiB steady state is in this number too: it is the practical
    ceiling of a single fused launch of that size, reported next to the roofline fraction."""
    import torch
    n = max(1, nbytes // 8)                       # floats per buffer
    nsets = min(32, max(2, int(-(-400e6 // nbytes))))
    a = [torch.empty(n, device=dev, dtype=torch.float32).normal_() for _ in range(nsets)]
    b = [torch.empty(n, device=dev, dtype=torch.float32) for _ in range(nsets)]
    for i in range(3):
        b[i % nsets].copy_(a[i % nsets])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        b[0].copy_(a[0])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for i in range(K):
            b[i % nsets].copy_(a[i % nsets])
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / K)
    ms = sorted(ts)[len(ts) // 2]
    peak, _ = measured_peak_gbs()
    gbs = 2 * n * 4 / (ms * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return {"ms_per_launch": ms, "achieved": gbs, "unit": "GB/s", "frac_of_peak": gbs / peak, "bytes_per_launch": 2 * n * 4,
            "what": "torch copy_ of the same number of bytes per launch (half read, half written), graph-replayed"}


def time_ops(name, dev, K, reps=3):
    """The path's other operators at a BASELINE shape (SURVEY.md 8f-1/2): the residual-minimisation form
    (forward operator pass + the backward operator pass, `resmin*`) and the un-fused
    gauss_pt_evaluation (`gp_eval*`, write-bound), graph-replayed like the headline.
    Returns {ms_per_step, bytes (algorithmic, per step), value GDOF/s}."""
    import torch
    from diffnet_b200 import ops
    kind, base = name.split(":")
    nsd, size, B, _, _ = WORKLOADS[base]
    fem = make_fem(base)
    dof = B * size ** nsd
    nsets = min(16, max(2, int(-(-400e6 // (dof * 24)))))
    sets = [make_inputs(base, dev, seed=777 + i) for i in range(nsets)]
    if kind == "resmin":
        jac = (0.5 * fem.h) ** nsd

        def step(i):
            s = sets[i % nsets]
            kw = {k: v for k, v in call_kwargs(s).items() if k in ("nu", "f", "dirichlet")}
            _, R = ops.residual_raw(fem.geometry, s["u"], jac=jac, apply_masks_to_input=True, **kw)
            kwb = {k: v for k, v in kw.items() if k in ("nu", "dirichlet")}
            return ops.residual_raw(fem.geometry, R, jac=jac, apply_masks_to_input=False, **kwb)
        nin = 5 if nsd == 2 else len(sets[0]["_fields"])                # 2-D: u, nu, bc1, bc2, f
        nbytes = dof * 4 * ((nin + 1) + (nin - 1 + 1))                   # pass 1: fields -> R; pass 2: R, nu, masks -> K R
    else:
        ngp = 2 ** nsd
        nel = B * (size - 1) ** nsd
        nbytes = dof * 4 + nel * ngp * 4
        if kind == "gp_eval_adj":          # the transpose: reads the cotangent at the Gauss points, writes the nodes
            cots = [torch.randn((B, ngp) + fem.geometry.elems, device=dev) for _ in range(max(2, min(nsets, 4)))]

            def step(i):
                return ops._gp_adj_raw(fem.geometry, cots[i % len(cots)], 0)
        else:
            def step(i):
                return ops._gp_raw(fem.geometry, sets[i % nsets]["u"], 0)
    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step(0)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for i in range(K):
            step(i)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / K)
    ms = sorted(ts)[len(ts) // 2]
    peak, _ = measured_peak_gbs()
    ach = nbytes / (ms * 1e-3) / 1e9
    return {"value": dof / (ms * 1e-3) / 1e9, "unit": "GDOF/s", "ms_per_step": ms, "algorithmic_bytes_per_step": nbytes,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak},
            "launches_per_step": 2 if kind == "resmin" else 1,
            "desc": ("residual form: operator pass + backward operator pass, " if kind == "resmin"
                     else "gauss_pt_evaluation (un-fused, N table), " if kind == "gp_eval"
                     else "adjoint of gauss_pt_evaluation (its autograd backward, N table), ") + WORKLOADS[base][4]}


OPS_POINTS = ["resmin:poisson2d_param_256_b64", "resmin:poisson3d_param_64_b16",
              "gp_eval:poisson2d_param_256_b64", "gp_eval:poisson3d_param_64_b16",
              "gp_eval_adj:poisson2d_param_256_b64", "gp_eval_adj:poisson3d_param_64_b16"]


def point_of(name, res, peak, clock_mhz=None):
    """One entry of `points`: a BASELINE config (or named roofline point) measured like the headline."""
    nsd, size, B, bpd, desc = WORKLOADS[name]
    dof = B * size ** nsd
    ms = res["ms_step"]
    val = dof / (ms * 1e-3) / 1e9
    ach = val * bpd
    fp32_peak = 148 * 128 * 2 * (clock_mhz or 1965.0) * 1e6 / 1e12      # TFLOP/s, FMA = 2
    tr = measured_traffic(name) or {}
    return {"value": val, "unit": "GDOF/s", "ms_per_step": ms, "bytes_per_dof": bpd,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_launch": dof * bpd, "traffic": tr.get("bytes"),
                         "traffic_read": tr.get("dram_read"), "traffic_write": tr.get("dram_write"),
                         "traffic_source": tr.get("source")},
            "secondary": {"bound": "fp32_pipe", "achieved": val * FLOPS_PER_DOF[nsd] / 1e3, "unit": "TFLOP/s",
                          "peak": fp32_peak, "frac": val * FLOPS_PER_DOF[nsd] / 1e3 / fp32_peak,
                          "algorithmic_flops_per_dof": FLOPS_PER_DOF[nsd]},
            "kernel": "k_fem2d_tma" if nsd == 2 else "k_fem3d_tma", "launch": res["mode"], "desc": desc}


POINTS = ["poisson2d_512_b16", "ibn2d_512_b16", "poisson3d_param_64_b16", "poisson3d_128_b1", "poisson3d_256_b1",
          "poisson2d_64_b1", "mms2d_fgp_256_b64", "mms3d_fgp_64_b16"]


# ------------------------------------------------------------------------------------ oracle legs
def oracle_step_time(name, sample_B, threads, repeats=8):
    """fwd+bwd of the oracle (reference conv path restated) on the CPU; best of `repeats`."""
    import torch
    from oracle import losses as OL
    from oracle.fem import Q1Oracle
    nsd, size, B, _, _ = WORKLOADS[name]
    torch.set_num_threads(threads)
    d = make_inputs_cpu(name, sample_B)
    o = Q1Oracle(nsd=nsd, domain_size=size)
    kw = call_kwargs(d)
    best = float("inf")
    for i in range(repeats + 1):
        u = d["u"].clone().requires_grad_(True)
        t0 = time.perf_counter()
        loss = OL.energy_loss(o, u, **kw)
        loss.backward()
        dt = time.perf_counter() - t0
        if i > 0:
            best = min(best, dt)
    dof = sample_B * size ** nsd
    return best, dof


def oracle_on_gpu_time(name, dev, repeats=5):
    """The reference's own path (conv2d/3d per Gauss point + pointwise + autograd, restated by the
    oracle) executed on THIS GPU through cuDNN with TF32 off: what a DiffNet user gets on a B200
    today.  A reported baseline like `cpu_baseline`, never the product path."""
    import torch
    from oracle import losses as OL
    from oracle.fem import Q1Oracle
    nsd, size, B, _, _ = WORKLOADS[name]
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    o = Q1Oracle(nsd=nsd, domain_size=size)
    for n in ("N_gp", "dN_x_gp", "dN_y_gp", "dN_z_gp"):
        setattr(o, n, [w.to(dev) for w in getattr(o, n)])
    o.gpw = o.gpw.to(dev)
    d = make_inputs(name, dev, seed=99)
    kw = call_kwargs(d)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = float("inf")
    for i in range(repeats + 2):
        u = d["u"].clone().requires_grad_(True)
        torch.cuda.synchronize()
        e0.record()
        OL.energy_loss(o, u, **kw).backward()
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            best = min(best, e0.elapsed_time(e1))
    del d, kw, u
    torch.cuda.empty_cache()
    return best * 1e-3, B * size ** nsd


def make_inputs_cpu(name, sample_B):
    import torch
    nsd, size, B, _, _ = WORKLOADS[name]
    saved = WORKLOADS[name]
    WORKLOADS[name] = (nsd, size, sample_B) + saved[3:]
    try:
        return make_inputs(name, torch.device("cpu"), seed=99)
    finally:
        WORKLOADS[name] = saved


def cpu_sample_batch(name):
    nsd, size, B, _, _ = WORKLOADS[name]
    dof_budget = 4.2e6 if nsd == 2 else 2.2e6    # ~1-4 s per oracle step on a few dozen cores
    return max(1, min(B, int(dof_budget // (size ** nsd)) or 1))


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port of DiffNetFEM.py + loss body; the
    reference is Python and /root/reference does not exist on the GPU box)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    nsd, size, B, bpd, desc = WORKLOADS[name]
    threads = os.cpu_count() or 1
    sB = cpu_sample_batch(name)
    torch.set_num_threads(threads)
    from oracle import losses as OL
    from oracle.fem import Q1Oracle
    d = make_inputs_cpu(name, sB)
    o = Q1Oracle(nsd=nsd, domain_size=size)
    kw = call_kwargs(d)

    def step():
        u = d["u"].clone().requires_grad_(True)
        OL.energy_loss(o, u, **kw).backward()
    # bounded sample: shrink the batch until (K + W) steps fit in ~2 minutes of CPU time; K and W
    # stay what --steps and --warmup say, so at a batch of 1 the run may take longer than that
    step()
    t0 = time.perf_counter(); step(); t1 = time.perf_counter() - t0
    budget, K, W = 120.0, args.steps, args.warmup
    if t1 * (K + W) > budget and sB > 1:
        sB = max(1, int(sB * budget / (t1 * (K + W))))
        d = make_inputs_cpu(name, sB)
        kw = call_kwargs(d)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    dof = sB * size ** nsd
    val = dof * args.steps / dt / 1e9
    sample = f"B={sB} of {B} samples per step ({dof} DOF), fwd+bwd w.r.t. u, torch {torch.__version__} CPU"
    print(json.dumps({
        "impl": "reference", "metric": "FEM loss+grad throughput", "value": val, "unit": "GDOF/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(name, args.gpus),
        "run": {"cpu_sample": sample},
        "cpu_baseline": {"value": val, "unit": "GDOF/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "GDOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def numa_local(dev_index):
    """Before the pinned host buffers of the e2e leg are allocated: run this rank on the cores of the NUMA node its
    GPU hangs off and prefer that node's memory, so that eight ranks do not all stream their inputs out of one
    socket's DRAM.  Best effort (sysfs may not expose the topology in a VM, set_mempolicy may be filtered): what was
    done is returned for the JSON line, failures leave the process as it was."""
    info = {"node": None, "cpus": None, "mempolicy": None}
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        info["node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
            info["_prev_affinity"] = allowed
        info["cpus"] = len(use) if use else 0
        try:
            import ctypes
            libc = ctypes.CDLL(None, use_errno=True)
            mask = ctypes.c_ulong(1 << node)
            MPOL_PREFERRED, SYS_set_mempolicy = 1, 238          # x86-64
            rc = libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(64))
            info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
        except Exception as e:   # noqa: BLE001
            info["mempolicy"] = f"{type(e).__name__}"
    except Exception as e:   # noqa: BLE001
        info["error"] = f"{type(e).__name__}: {e}"
    return info


def numa_restore(info):
    """Undo numa_local once the pinned buffers exist (the CPU legs that follow want every core)."""
    try:
        prev = info.pop("_prev_affinity", None)
        if prev:
            os.sched_setaffinity(0, prev)
        if info.get("mempolicy") == "preferred":
            import ctypes
            ctypes.CDLL(None, use_errno=True).syscall(238, 0, None, ctypes.c_ulong(0))      # MPOL_DEFAULT
    except Exception:   # noqa: BLE001
        pass


# ------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    name = args.workload
    nsd, size, B, bpd, desc = WORKLOADS[name]
    dof_step = B * size ** nsd                     # per GPU per step
    step_bytes = dof_step * bpd
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    reps = args.reps
    res = time_workload(name, dev, 1234 + 17 * rank, K, W, reps, world, barrier, not args.no_graph,
                        keep_last=bool(args.dump_outputs))
    sets, fem, nsets, mode = res["sets"], res["fem"], res["nsets"], res["mode"]
    dumped = dump_outputs(args.dump_outputs, res.pop("last")) if args.dump_outputs and rank == 0 else None
    t = torch.tensor([res["ms_step"]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item())
    value = dof_step * world / (ms_step * 1e-3) / 1e9

    # ---- e2e: public API, pinned host inputs, H2D + launch + D2H(loss) every step
    numa = numa_local(local)
    hs = sets[0]
    host = [f.detach().cpu().pin_memory() for f in hs["_fields"]]
    devbuf = [torch.empty_like(f) for f in hs["_fields"]]
    h2d = sum(h.numel() * h.element_size() for h in host)

    def rebuild(fields):
        if nsd == 2:
            u, inputs, f = fields
            return u, dict(nu=inputs[:, 0:1], f=f, dirichlet=[(inputs[:, 1:2], 1.0), (inputs[:, 2:3], 0.0)])
        kw = dict(call_kwargs(hs))
        ordered = [t for t in hs["_fields"]]
        remap = {id(o): n for o, n in zip(ordered, fields)}
        def m(x):
            return remap.get(id(x), x)
        kw = {k: (m(v) if torch.is_tensor(v) else ([(m(a), b) for a, b in v] if k == "dirichlet" else v))
              for k, v in kw.items()}
        return m(hs["u"]), kw

    # double-buffered like any input pipeline: step i+1's H2D (copy stream) overlaps step i's launch and the
    # read-back of its loss; every step's copy and read-back are inside the timed region
    copy_stream = torch.cuda.Stream(device=dev)
    devsets = [devbuf, [torch.empty_like(f) for f in hs["_fields"]]]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    freed = [torch.cuda.Event(), torch.cuda.Event()]

    def start_copy(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[i % 2])            # the launch that last read this buffer set
            for h, d in zip(host, devsets[i % 2]):
                d.copy_(h, non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_step(i):
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(ready[i % 2])
        u, kw = rebuild(devsets[i % 2])
        loss, grad = fem.energy_loss_and_grad(u, **kw)
        freed[i % 2].record(cur)
        start_copy(i + 1)
        return float(loss)                          # D2H read of the step's result (syncs the compute stream)

    start_copy(0)
    for i in range(3):
        e2e_step(i)
    torch.cuda.synchronize()
    Ke = max(3, min(K, 20))
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    copy_stream.wait_event(g0)                      # the first timed copy starts inside the timed region
    start_copy(3)
    for i in range(3, 3 + Ke):
        e2e_step(i)                                 # H2D copies + launch + loss.item() (a sync) every step
    g1.record()
    torch.cuda.synchronize()
    te = torch.tensor([g0.elapsed_time(g1) * 1e-3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = dof_step * world * Ke / float(te.item()) / 1e9
    # ---- the same step with the inputs PRODUCED on the device (SURVEY.md 8f-3): what crosses PCIe is u (in
    # training it is the network's output and never leaves the device) and the 6 KL coefficients per sample
    # (KLSumStochastic / gen_input_calc.py restated as a kernel); nu, bc1, bc2, f are written by the producer
    e2e_prod = None
    if name == DEFAULT:
        try:
            from diffnet_b200.datasets import kl_inputs
            gco = torch.Generator(device="cpu").manual_seed(99 + rank)
            hco = (torch.rand(B, 6, generator=gco, dtype=torch.float64) * 6.0 - 3.0).pin_memory()
            dco = torch.empty(B, 6, dtype=torch.float64, device=dev)
            hu, du = host[0], devbuf[0]

            def prod_step():
                du.copy_(hu, non_blocking=True)
                dco.copy_(hco, non_blocking=True)
                inp, frc = kl_inputs(dco, size, 2, 0.5, None, dev)
                loss, grad = fem.energy_loss_and_grad(du, nu=inp[:, 0:1], f=frc,
                                                      dirichlet=[(inp[:, 1:2], 1.0), (inp[:, 2:3], 0.0)])
                return float(loss)
            for _ in range(3):
                prod_step()
            barrier()
            g0.record()
            for _ in range(Ke):
                prod_step()
            g1.record()
            torch.cuda.synchronize()
            tp = torch.tensor([g0.elapsed_time(g1) * 1e-3], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            hb = hu.numel() * 4 + hco.numel() * 8
            e2e_prod = {"value": dof_step * world * Ke / float(tp.item()) / 1e9, "unit": "GDOF/s",
                        "h2d_bytes_per_step": hb, "d2h_bytes_per_step": 4, "steps": Ke,
                        "note": "u + the KL coefficients from pinned host memory, nu/bc1/bc2/f written by the producer kernel "
                                "(dn_gen_kl_inputs_f32), fused launch, loss.item(): the step a DiffNet training loop runs "
                                "when its dataset lives on the device"}
        except Exception as e:   # noqa: BLE001
            e2e_prod = {"error": f"{type(e).__name__}: {e}"}
    # ---- opt-in compact ingestion (same loss, same fused kernel): the two Dirichlet masks shipped as uint8
    # (the op widens them on the device) and the all-zero source term as ONE broadcast image (stride_b = 0)
    e2e_compact = None
    if name == DEFAULT:
        try:
            hu, hin, hf = host
            h_nu = hin[:, 0:1].contiguous().pin_memory()
            h_m1 = (hin[:, 1:2] > 0.5).to(torch.uint8).contiguous().pin_memory()
            h_m2 = (hin[:, 2:3] > 0.5).to(torch.uint8).contiguous().pin_memory()
            h_f1 = hf[:1].contiguous().pin_memory()
            hostc = [hu, h_nu, h_m1, h_m2, h_f1]
            devc = [torch.empty_like(t, device=dev) for t in hostc]

            def compact_step():
                for h, d in zip(hostc, devc):
                    d.copy_(h, non_blocking=True)
                loss, grad = fem.energy_loss_and_grad(devc[0], nu=devc[1], f=devc[4],
                                                      dirichlet=[(devc[2], 1.0), (devc[3], 0.0)])
                return float(loss)
            for _ in range(3):
                compact_step()
            barrier()
            g0.record()
            for _ in range(Ke):
                compact_step()
            g1.record()
            torch.cuda.synchronize()
            tc = torch.tensor([g0.elapsed_time(g1) * 1e-3], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tc, op=dist.ReduceOp.MAX)
            hb = sum(t.numel() * t.element_size() for t in hostc)
            e2e_compact = {"value": dof_step * world * Ke / float(tc.item()) / 1e9, "unit": "GDOF/s",
                           "h2d_bytes_per_step": hb, "d2h_bytes_per_step": 4, "steps": Ke,
                           "h2d_gbs_per_gpu": hb * Ke / float(tc.item()) / 1e9,
                           "note": "opt-in: Dirichlet masks as uint8 (widened on the device by the op), the zero source term as "
                                   "one broadcast image; u and nu fp32 per sample; otherwise the e2e step"}
            del hostc, devc
        except Exception as e:   # noqa: BLE001
            e2e_compact = {"error": f"{type(e).__name__}: {e}"}
    del sets, res, devbuf, host, hs
    torch.cuda.empty_cache()
    copyref = None
    if world == 1:
        try:
            copyref = copy_reference(dev, step_bytes)
        except Exception as e:   # noqa: BLE001
            copyref = {"error": f"{type(e).__name__}: {e}"}
    numa_restore(numa)
    # ---- the other BASELINE configs and the north_star's named roofline points, measured the same way
    points = None
    if world == 1 and args.points and name == DEFAULT:
        peak0, _ = measured_peak_gbs()
        points = {}
        for pn in POINTS:
            try:
                r = time_workload(pn, dev, 4321, max(20, min(K, 100)), 5, 3)
                points[pn] = point_of(pn, r, peak0)
                del r
                torch.cuda.empty_cache()
                pnsd, psize, pB, pbpd, _ = WORKLOADS[pn]
                cr = copy_reference(dev, pB * psize ** pnsd * pbpd)
                points[pn]["roofline"]["same_bytes_copy"] = cr
                points[pn]["roofline"]["frac_of_same_bytes_copy"] = points[pn]["roofline"]["achieved"] / cr["achieved"]
                if pn.startswith("mms"):       # the same call with f_gp read by the general kernels every step
                    from diffnet_b200 import ops as _ops
                    _ops.USE_LOAD_VECTOR = False
                    try:
                        r = time_workload(pn, dev, 4321, 20, 5, 3)
                        points[pn]["f_gp_in_general_kernel_ms"] = r["ms_step"]
                        points[pn]["note"] = ("f_gp is assembled ONCE into a load vector b (dn_fem_load_vector_f32, cached "
                                              "per tensor version); the timed step streams b.  f_gp_in_general_kernel_ms: the "
                                              "same call with f_gp read at the Gauss points every step (DN_LOAD_VECTOR=0)")
                        del r
                    finally:
                        _ops.USE_LOAD_VECTOR = True
            except Exception as e:   # noqa: BLE001  (the headline must still be printed)
                points[pn] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
        for pn in OPS_POINTS:
            try:
                points[pn] = time_ops(pn, dev, 20)
            except Exception as e:   # noqa: BLE001
                points[pn] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()
    clocks = sampler.stop() if rank == 0 else None
    if points and clocks and clocks.get("sm_mhz"):
        for v in points.values():
            if "secondary" in v:
                pk = 148 * 128 * 2 * clocks["sm_mhz"] * 1e6 / 1e12
                v["secondary"]["peak"], v["secondary"]["frac"] = pk, v["secondary"]["achieved"] / pk
                v["secondary"]["clock_mhz"] = clocks["sm_mhz"]
    train = None
    if args.train_steps > 0 and name in ("poisson2d_param_256_b64", "poisson3d_param_64_b16"):
        try:
            train = train_step_rate(name, dev, world, rank, args.train_steps, 5)
        except Exception as e:   # noqa: BLE001  (the FEM line must still be printed)
            train = {"error": f"{type(e).__name__}: {e}"}
    # ---- N > 1: the one path with a real exchange step (256^3 field in z-slabs, peer-memory halos)
    slab = None
    if world > 1 and args.slab and name == DEFAULT:
        try:
            slab = slab_measure(args, world, rank, dev, steps=max(20, min(K, 100)))
        except Exception as e:   # noqa: BLE001
            slab = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        achieved = step_bytes / (ms_step * 1e-3) / 1e9
        cpu = None
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            sB = cpu_sample_batch(name)
            best, dof = oracle_step_time(name, sB, threads)
            cpu = {"value": dof / best / 1e9, "unit": "GDOF/s", "cores": threads, "kind": "port",
                   "sample": f"oracle fwd+bwd on B={sB} of {B} samples ({dof} DOF), best of 8, torch {torch.__version__} CPU"}
            if name != "poisson3d_256_b1":      # the conv path materialises ~20 GB of Gauss-point tensors at 256^3
                try:
                    tg, dg = oracle_on_gpu_time(name, dev)
                    cpu["same_path_on_this_gpu"] = {
                        "value": dg / tg / 1e9, "unit": "GDOF/s", "ms_per_step": tg * 1e3,
                        "note": "the reference conv path (oracle port) on this B200 via cuDNN, TF32 off, full batch, "
                                "best of 5 -- a baseline, not the product path"}
                except Exception as e:   # noqa: BLE001
                    cpu["same_path_on_this_gpu"] = {"error": f"{type(e).__name__}: {e}"}
        tr = measured_traffic(name) or {}
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        fp32_peak = 148 * 128 * 2 * mhz * 1e6 / 1e12
        line = {
            "metric": "FEM loss+grad throughput", "value": value, "unit": "GDOF/s", "n_gpus": world,
            "steps": K, "warmup": max(W, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(name, world),
            "run": {"launch": mode,
                    "timing": f"CUDA events around {K} steps, median of {reps} repetitions, max over ranks"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": tr.get("bytes"),
                         "traffic_read": tr.get("dram_read"), "traffic_write": tr.get("dram_write"),
                         "traffic_note": tr.get("note"), "traffic_source": tr.get("source"),
                         "peak_source": peak_src, "bytes_per_dof": bpd,
                         "algorithmic_bytes_per_launch": step_bytes,
                         "same_bytes_copy": copyref,
                         "frac_of_same_bytes_copy": (achieved / copyref["achieved"]) if copyref and "achieved" in copyref else None,
                         "kernel": "k_fem2d_tma" if nsd == 2 else "k_fem3d_tma",
                         "secondary": {"bound": "fp32_pipe", "unit": "TFLOP/s",
                                       "achieved": value / world * FLOPS_PER_DOF[nsd] / 1e3, "peak": fp32_peak,
                                       "frac": value / world * FLOPS_PER_DOF[nsd] / 1e3 / fp32_peak,
                                       "algorithmic_flops_per_dof": FLOPS_PER_DOF[nsd],
                                       "note": "148 SMs x 128 lanes x 2 x the SM clock under load; 3-D is bound here "
                                               "(register-operand dispatch), 2-D by HBM"}},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "GDOF/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "steps": Ke, "h2d_gbs_per_gpu": h2d * Ke / float(te.item()) / 1e9, "numa": numa,
                    "note": "pinned host -> device copy of all input fields + fused launch + loss.item() every step, double-buffered (the next step's copy overlaps this step's launch and read-back); CUDA events around the steps, max over ranks"},
            "e2e_compact_inputs": e2e_compact,
            "e2e_device_producers": e2e_prod,
            "gpu_launches": K,
            "clocks": clocks,
            "train": train,
            "points": points,
            "slab": slab,
        }
        if dumped is not None:
            line["dumped_outputs"] = dumped
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------ train step
def train_step_rate(name, dev, world, rank, steps, warmup):
    """Full training step of the parametric config: UNet forward + fused FEM loss + backward +
    DDP gradient all-reduce (NCCL) + Adam; batch per GPU fixed (weak scaling); synthetic inputs
    resident on the device; CUDA events around `steps` steps, max over ranks."""
    import torch
    import torch.distributed as dist
    from diffnet_b200.networks import UNet
    from diffnet_b200.poisson import PoissonIBN3D, PoissonParametric2D
    from diffnet_b200.synthetic import poisson2d_parametric_batch, poisson3d_parametric_batch
    nsd, size, B, _, _ = WORKLOADS[name]
    torch.manual_seed(0)
    if nsd == 2:
        net = UNet(3, 1).to(dev)
        mod = PoissonParametric2D(net, domain_size=size, batch_size=B, learning_rate=3e-4)
        _, inputs, f = poisson2d_parametric_batch(B, size, dev, seed=4321 + rank)
        batch = (inputs, f)
    else:
        net = UNet(1, 1, nd=3).to(dev)
        mod = PoissonIBN3D(net, domain_size=size, batch_size=B, learning_rate=3e-4)
        _, src, sink, f = poisson3d_parametric_batch(B, size, dev, seed=4321 + rank)
        batch = (src, sink, f)
    mod.to(dev)
    nparams = sum(p.numel() for p in net.parameters())
    if world > 1:
        mod.network = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index],
                                                               gradient_as_bucket_view=True)
    opt = mod.configure_optimizers()[0][0]
    mod.train()

    def step():
        opt.zero_grad(set_to_none=True)
        loss = mod.training_step(batch, 0)
        loss.backward()
        opt.step()
        return loss

    for _ in range(max(warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    return {"steps_per_s": 1e3 / ms, "samples_per_s": 1e3 / ms * B * world, "ms_per_step": ms, "steps": steps,
            "batch_per_gpu": B, "network": f"UNet nd={nsd} ({nparams} params)", "loss": float(loss),
            "note": "UNet fwd + fused FEM loss + bwd + DDP all-reduce (NCCL) + Adam; fp32; weak scaling"}


# ------------------------------------------------------------------------------------ z-slab arm
def slab_measure(args, world, rank, dev, steps=None, workload="poisson3d_256_slab"):
    """One 256^3 field over all ranks (SURVEY.md 8e): per step = halo exchange of u + fused kernel on
    the slab + scalar loss all-reduce.  Strong scaling.  Needs an initialised process group when
    world > 1.  Returns the result dict on rank 0 (None elsewhere), including a bit-exactness check
    of the loss against the single-kernel value where that is cheap (world == 1 trivially true)."""
    import torch
    import torch.distributed as dist
    from diffnet_b200 import ops
    from diffnet_b200.slab import ZSlabPoisson3D, make_slab
    nsd, N, _, bpd, desc = WORKLOADS[workload]
    h = 1.0 / (N - 1)
    geom = ops.Geometry(3, N, N, N, h, h, h, 2)
    sp = ZSlabPoisson3D(geom, transport=args.transport)
    sl = make_slab(N, world, rank)
    nl = sl.hi - sl.lo
    g = torch.Generator(device=dev).manual_seed(1234 + sl.lo)
    # synthetic slab-local fields (solve_in_object_3d.py:37-62 shapes: nu = object mask, bc1 = outside, f = 500)
    zz = torch.arange(sl.lo, sl.hi, device=dev).float()[:, None, None] / (N - 1) - 0.5
    yy = torch.arange(N, device=dev).float()[None, :, None] / (N - 1) - 0.5
    xx = torch.arange(N, device=dev).float()[None, None, :] / (N - 1) - 0.5
    inside = ((xx ** 2 + yy ** 2 + zz ** 2) < 0.16).float()
    nsets = 4          # rotate 4 slabs: the per-rank working set must not live in the 126 MB L2
    us = [torch.randn(nl, N, N, device=dev, generator=g) for _ in range(nsets)]
    sp.set_fields(nu=inside, f=torch.full_like(inside, 500.0), dirichlet=[(1.0 - inside, 0.0)],
                  already_local=True, c_k=0.5)
    K, W = steps or args.steps, max(args.warmup, 3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(step):
        for i in range(W):
            step(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for i in range(K):
            out = step(i)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / K, out

    # (1) the linked step: ONE launch per rank (puts + flag waits + FEM kernel + loss push), graph-replayed
    linked_ms, linked_mode, loss_linked = None, None, None
    if world > 1 and args.transport == "peer":
        try:
            rp = sp.capture(us, linked=True) if not args.no_graph else None
            linked_mode = "cuda_graph (one linked launch per step)" if rp is not None else "eager (one linked launch per step)"
            linked_ms, _ = timed((lambda i: rp()) if rp is not None else (lambda i: sp.step_linked(us[i % nsets])))
            loss_linked = float(sp.global_loss())
        except Exception as e:   # noqa: BLE001
            linked_mode = f"failed: {type(e).__name__}: {e}"
            torch.cuda.synchronize()
    # (2) separate launches: halo put/wait kernels (or NCCL) + FEM kernel + peer all-reduce of the loss
    kw = dict(zero_halo_grad=False, overlap=args.overlap and args.transport != "peer")
    mode = "eager"
    replays = None
    # NCCL point-to-point inside a captured graph hung on this stack: graphs need the peer transport for N > 1
    if not args.no_graph and (world == 1 or args.transport == "peer"):
        try:
            replays = sp.capture(us, **kw)
            mode = "cuda_graph (halo put/wait + FEM kernel + peer all-reduce captured)"
        except Exception as e:   # noqa: BLE001
            replays, mode = None, f"eager (graph capture failed: {type(e).__name__}: {e})"
            torch.cuda.synchronize()
    sep_ms, (loss, grad) = timed((lambda i: replays()) if replays is not None
                                 else (lambda i: sp.loss_and_grad(us[i % nsets], **kw)))
    ms = linked_ms if linked_ms is not None else sep_ms
    dof = N ** 3
    # exchange alone (put + wait of both halo planes), same launch path, for the step's timeline
    xms = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        e0.record()
        for i in range(20):
            sp.exchange_halos(us[i % nsets])
        e1.record()
        torch.cuda.synchronize()
        tx = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        dist.all_reduce(tx, op=dist.ReduceOp.MAX)
        xms = float(tx.item()) / 20
    # the two paths on the SAME slab: global loss (different summation of the partials: tolerance) and
    # owned gradient (bit for bit)
    parity_check = None
    if world > 1 and linked_ms is not None:
        o0, o1 = sp.slab.own_local
        l_sep, g_sep = sp.loss_and_grad(us[0], **kw)
        g_sep = g_sep.clone()
        _, g_l = sp.step_linked(us[0])
        l_link = sp.global_loss()
        eq = torch.tensor([1.0 if torch.equal(g_l[o0:o1], g_sep[o0:o1]) else 0.0], device=dev)
        dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        parity_check = {"loss_rel_diff": abs(float(l_link) - float(l_sep)) / max(abs(float(l_sep)), 1e-30),
                        "owned_grad_bit_equal_all_ranks": bool(eq.item() == 1.0)}
    timed_out = bool(sp._peer_halo.timed_out()) if getattr(sp, "_peer_halo", None) is not None else False
    if rank != 0:
        return None
    peak, peak_src = measured_peak_gbs()
    value = dof / (ms * 1e-3) / 1e9
    achieved = dof * bpd / (ms * 1e-3) / 1e9 / world
    return {"workload": workload, "desc": desc, "value": value, "unit": "GDOF/s", "n_gpus": world, "scaling": "strong",
            "ms_per_step": ms, "steps": K, "exchange_ms_eager": xms, "slab_planes_rank0": nl,
            "launch": linked_mode if linked_ms is not None else mode,
            "separate_launches": {"ms_per_step": sep_ms, "value": dof / (sep_ms * 1e-3) / 1e9, "launch": mode,
                                  "loss": float(loss)},
            "linked": {"ms_per_step": linked_ms, "launch": linked_mode, "global_loss": loss_linked,
                       "vs_separate_launches": parity_check},
            "transport": ("NVLink peer-memory put/wait kernels (CUDA IPC)" if args.transport == "peer"
                          else "ncclSend/Recv") + (" overlapped with the interior planes" if args.overlap else ""),
            "nvlink_bytes_per_step_per_rank": (2 if world > 1 else 0) * N * N * 4,
            "roofline_per_gpu": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                                 "frac": achieved / peak, "bytes_per_dof": bpd, "kernel": "k_fem3d_tma"},
            "loss": float(loss), "device_wait_timed_out": timed_out,
            "l2": f"{nsets} rotating slabs x {nl * N * N * bpd / 1e6:.0f} MB per rank (static fields shared)"}


def run_slab(args):
    """--workload poisson3d_256_slab: the z-slab arm on its own (one JSON line)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    r = slab_measure(args, world, rank, dev)
    if rank == 0:
        name = args.workload
        print(json.dumps({
            "metric": "FEM loss+grad throughput", "value": r["value"], "unit": "GDOF/s", "n_gpus": world,
            "steps": r["steps"], "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "desc": r["desc"], "grid": [256, 256, 256],
                       "slab_planes_rank0": r["slab_planes_rank0"], "launch": r["launch"], "l2": r["l2"],
                       "timing": f"CUDA events around {r['steps']} steps, max over ranks",
                       "parallelism": f"z-slab x{world}: {r['transport']} for the 2 halo planes + loss all-reduce per step"},
            "roofline": dict(r["roofline_per_gpu"], traffic=None,
                             note="per-GPU: algorithmic bytes of the rank's owned planes / step time"),
            "cpu_baseline": None, "e2e": None, "gpu_launches": r["steps"], "clocks": None, "loss": r["loss"],
            "slab": r}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT, choices=sorted(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--transport", default="peer", choices=["peer", "nccl"],
                    help="z-slab arm: halo transport (our NVLink peer-memory kernels, or NCCL send/recv)")
    ap.add_argument("--overlap", action="store_true",
                    help="z-slab arm: interior planes while the halos are in flight (3 launches instead of 1)")
    ap.add_argument("--no-points", dest="points", action="store_false",
                    help="skip the extra BASELINE configs / roofline points reported under `points` (N = 1)")
    ap.add_argument("--no-slab", dest="slab", action="store_false",
                    help="skip the 256^3 z-slab arm reported under `slab` (N > 1)")
    ap.add_argument("--train-steps", type=int, default=20,
                    help="also time this many full training steps (UNet + loss + DDP + Adam); 0 = skip")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write (loss, grad) of the last timed step of rank 0 as DIR/loss.npy and DIR/grad.npy "
                         "(a seeded sample of grad when both exceed 60 MB); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload == "poisson3d_256_slab"):
        ap.error("--dump-outputs covers the fused-kernel arm (--impl ours) of the batched workloads")
    if args.impl == "reference":
        if args.workload == "poisson3d_256_slab":
            args.workload = "poisson3d_256_b1"
        run_reference(args)
    elif args.workload == "poisson3d_256_slab":
        run_slab(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
