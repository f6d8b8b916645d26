#!/usr/bin/env python
"""Benchmark of the SchNetPack message-passing hot path on B200 (driver contract: one JSON line on rank 0).

    python bench.py --gpus 1 --steps 20 --warmup 5                  # CUDA path (this repo)
    python bench.py --impl reference --gpus 1 --steps 5 --warmup 1  # reference arm: CPU path on the host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...            # weak scaling: one batch per rank, no collective
    torchrun --nproc-per-node N ... bench.py --gpus N --config cfg5  # STRONG scaling: one 262144-atom periodic box split
                                                                     # into N slabs, NCCL halo exchange of ghost rows

Workload (BASELINE.json configs[1]): MD17 aspirin x 256, PaiNN F=128 T=3 (20 Gaussian RBF, cosine cutoff 5 A),
energy + forces.  One *step* = one full evaluation ``model(inputs)`` of the whole batch (256 molecule-evals).
``value`` = molecule-evals/s with inputs resident in HBM; ``e2e`` = the same call fed from pinned HOST buffers with the
H2D copies of the batch and the D2H read of energy+forces inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from schnetpack_b200 import synthetic as S  # noqa: E402

METRIC = "energy+force evals/s"
UNIT = "molecule-evals/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload(name: str, rank: int, batch: int | None):
    kw = {}
    if name in ("cfg1", "cfg2", "cfg3") and batch is not None:
        kw["batch"] = batch
    if name in ("cfg2", "cfg3"):
        kw["seed"] = rank
    spec, data = S.make_config(name, **kw)
    return spec, data


def n_systems(data):
    return int(data[S.n_atoms].shape[0])


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write the outputs of the last timed step as ``out_dir/<name>.npy`` (fp32 as computed, fp64 kept), so that two
    builds run with the same arguments -- hence the same seeded inputs and weights -- can be compared output for output.
    Should they exceed 64 MB together, every array keeps a fixed, seeded sample of its rows."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT and a.ndim > 0:
            keep = max(1, int(a.shape[0] * DUMP_LIMIT // total))
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------- algorithmic bytes
def edge_kernel_bytes(E, N, F, has_mu, backward):
    """SURVEY.md §8(d) 'no-reuse gather model' per launch of the fused PaiNN edge kernel.
    forward : E*(8+8+12 + 4*3F [x_j] + 4*3F [mu_j]) + N*(4*4F read q,mu + 4*4F write)      = E*3100 + N*4096 (F=128)
    backward: E*(28 + 2*4*3F regather + 2*4*3F sender-grad accumulate + 12) + N*(2*4*4F)   = E*6184 + N*4096
    first block (mu == 0): no mu_j gather and no mu-dependent third."""
    if not backward:
        per_e = 28 + 4 * 3 * F + (4 * 3 * F if has_mu else 0)
        per_n = 4 * 4 * F * 2 if has_mu else 4 * F + 4 * 4 * F
    else:
        per_e = 28 + 2 * 4 * 3 * F + (2 * 4 * 3 * F if has_mu else 0) + 12
        per_n = 2 * 4 * 4 * F
    return E * per_e + N * per_n


class ClockSampler:
    """SM clock + throttle reasons of the benchmarked GPU, sampled WHILE the warm-up and the timed steps run: NVML in a
    thread (one query every 5 ms: a 50 ms timed region still gets samples), `nvidia-smi -lms` only when NVML is missing."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                    ("sw_power_cap", 0x4))

    def __init__(self, gpu_index: int):
        self.p = self.f = self.thread = None
        self.sm, self.reasons, self.mx = [], set(), None
        try:
            import threading

            import pynvml

            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + uuid)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.stop_flag = threading.Event()
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.QUERY}",
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def _poll(self):
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                bits = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for name, bit in self.NVML_REASONS:
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_flag.wait(0.005)

    def mark(self):
        """Start of the timed region: samples from here on are the reported ones (warm-up samples only if there are none)."""
        self.mark_at = len(self.sm)

    def stop(self):
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            sm = self.sm[getattr(self, "mark_at", 0):] or self.sm
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------- reference (CPU) arm
def reference_engine(spec, params, data, device=None):
    """(callable evaluating one full batch, kind).  The reference's OWN modules (oracle/ref_loader.py: /root/reference or the
    vendored byte-identical copy oracle/_ref) when present -> kind "reference"; otherwise the restatement
    oracle/spk_oracle.py (the same ATen op sequence) -> kind "port"."""
    from oracle import ref_loader as rl

    if rl.available():
        model = rl.build_from_spec(spec, params, torch.float32, device)
        x0 = {}
        for k, v in data.items():
            t = torch.as_tensor(v)
            if t.is_floating_point():
                t = t.float()
            x0[k] = t.to(device) if device is not None else t
        forces = bool(spec.get("forces", True))

        def run():
            x = {k: (v.detach().clone() if v.is_floating_point() else v) for k, v in x0.items()}   # fresh leaves per call
            if "_Rij" in x:
                x = model.representation(x)
                return model.output_modules[0](x)
            return model(x)

        _ = forces
        return run, "reference"
    from oracle import spk_oracle as O

    if device is None:
        return (lambda: O.energy_forces(spec, params, data, dtype=torch.float32)), "port"
    p_dev = O.to_torch(params, torch.float32, device)
    x_dev = O.to_torch(data, torch.float32, device)
    return (lambda: O.energy_forces(spec, p_dev, x_dev, device=device)), "port"


def cpu_eval_time(run, steps, warmup, threads):
    torch.set_num_threads(threads)
    ts = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if it >= warmup:
            ts.append(dt)
    return ts


def best_thread_count(run):
    """BASELINE.md section 3 asks for torch.set_num_threads(os.cpu_count()); the reference's eager CPU path scales badly
    past a few dozen threads on these small ops (128 threads were 13x slower than 8 on the round-1 box), so the arm is
    given the thread count it is FASTEST with (favours the reference): probe 8/16/32/64/all once each, keep the best.
    Returns (threads, seconds_per_eval_at_that_count)."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} or {cores})
    best = None
    first = True
    for c in cands:
        t = min(cpu_eval_time(run, 1, 1 if first else 0, c))
        first = False
        if best is None or t < best[1]:
            best = (c, t)
        elif t > 1.5 * best[1]:
            break
    return best


def cpu_sample(args):
    """The bounded CPU sample of a workload: (spec, data, scale, description).  cfg5's 262144-atom box does not fit a CPU
    reference evaluation in minutes: the CPU arm evaluates a 16384-atom periodic box of the same density and model and its
    rate is scaled by the atom ratio (labelled as such)."""
    if args.config == "cfg5":
        n_sub = 16384
        spec, data = S.make_config("cfg4", n_atoms_total=n_sub)
        n_full = args.atoms or 262144
        return spec, data, n_sub / n_full, (f"{n_sub}-atom periodic sub-box of the same density / model, rate scaled by "
                                            f"{n_sub}/{n_full} atoms")
    spec, data = workload(args.config, 0, args.batch)
    return spec, data, 1.0, "the full batch"


def config_dict(args, world, B, N, E, F, T):
    """ONE description of the workload, identical in both arms (the driver compares them)."""
    spatial = args.config == "cfg5"
    return {"workload": f"{args.config}: {S.CONFIGS[args.config]['desc']}", "systems_per_gpu": (1 if spatial else B),
            "atoms": N, "edges": E, "n_atom_basis": F, "n_interactions": T,
            "parallelism": (f"spatial x{world}: one periodic box in {world} slab(s), NCCL halo exchange of ghost rows"
                            if spatial else f"batch-sharded x{world}"),
            "weights": "seeded xavier-uniform (synthetic.init_params)",
            "timing": {"b200": "CUDA events per step on the launch stream, 256 MiB device memset between timed steps "
                               "(outside the event intervals); step = CUDA-graph replay of model(inputs) on the resident "
                               "batch (cfg5: eager per-block pipeline, tables exceed L2)",
                       "reference": "time.perf_counter per full evaluation of the reference modules on the host cores"}}


def run_reference(args, rank, world):
    """The reference's CPU path: the UNMODIFIED reference modules (kind 'reference', oracle/_ref) -- or the oracle port if
    they are absent -- timed on the host cores.  Rank 0 only."""
    if rank != 0:
        return
    spec, data, scale, what = cpu_sample(args)
    params = S.init_params(spec, seed=0)
    run, kind = reference_engine(spec, params, data)
    cores, _ = best_thread_count(run)
    ts = cpu_eval_time(run, args.steps, args.warmup, cores)
    B = n_systems(data)
    N_s, E_s = int(data[S.Z].shape[0]), int(data[S.idx_i].shape[0])
    if args.config == "cfg5":
        N, E = args.atoms or 262144, int(round(E_s / scale))
    else:
        N, E = N_s, E_s
    ms = 1e3 * float(np.mean(ts)) / scale
    v = B * scale / float(np.mean(ts))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.config == "cfg5" else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, args.gpus, B, N, E, spec["n_atom_basis"], spec["n_interactions"]),
        "edge_msgs_per_s": E_s * spec["n_interactions"] / float(np.mean(ts)),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{args.steps} evaluations of {what} ({B} systems, {N_s} atoms, {E_s} edges) after "
                                   f"{args.warmup} warm-up, "
                                   + ("the reference's own modules (oracle/ref_loader.py)" if kind == "reference"
                                      else "oracle/spk_oracle.py (same ATen op sequence as the reference)")
                                   + f", fp32, torch.set_num_threads({cores}) = fastest of 8/16/32/64/{os.cpu_count()} "
                                     f"probed; median {1e3 * float(np.median(ts)):.1f} ms, min {1e3 * float(np.min(ts)):.1f} ms"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(args):
    spec, data, scale, what = cpu_sample(args)
    params = S.init_params(spec, seed=0)
    run, kind = reference_engine(spec, params, data)
    cores, _ = best_thread_count(run)
    ts = cpu_eval_time(run, 3, 0, cores)
    B = n_systems(data)
    return {"value": B * scale / float(np.mean(ts)), "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"3 evaluations of {what} ({B} systems, {int(data[S.Z].shape[0])} atoms, "
                      f"{int(data[S.idx_i].shape[0])} edges), "
                      + ("the reference's own modules (oracle/ref_loader.py)" if kind == "reference"
                         else "oracle/spk_oracle.py (the reference's ATen op sequence)")
                      + f", fp32, {cores} threads (fastest of 8/16/32/64/{os.cpu_count()} probed on this host); "
                        f"mean {1e3 * float(np.mean(ts)):.0f} ms"}


def eager_gpu_leg(spec, params, data, dev, B, n_it=10):
    """The reference's own single-GPU eager PyTorch path (modules .to(cuda), cuBLAS SGEMM, index_select / index_add_ atomics,
    autograd backward) on the same B200, inputs resident: the denominator of the north-star's >= 5x target."""
    try:
        run, kind = reference_engine(spec, params, data, device=dev)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_it):
            run()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / n_it
        return {"value": B / dt, "unit": UNIT, "ms_per_step": 1e3 * dt, "kind": kind,
                "what": "the reference's modules in eager PyTorch on the same B200 (wall clock, synchronised), inputs resident"}
    except Exception as exc:  # pragma: no cover
        return {"error": repr(exc)[:200]}


# ------------------------------------------------------------------------------------------------- CUDA arm
def run_cuda(args, rank, world, local_rank):
    import schnetpack_b200 as sb
    from schnetpack_b200 import _lib, ops
    from schnetpack_b200.model import batch_to_device, from_spec

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"          # NCCL's version banner goes to stdout: keep the ONE JSON line clean
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=dev)

    spec, data = workload(args.config, rank, args.batch)
    params = S.init_params(spec, seed=0)
    model = from_spec(spec, params, dev)
    B, N, E = n_systems(data), int(data[S.Z].shape[0]), int(data[S.idx_i].shape[0])
    F, T = spec["n_atom_basis"], spec["n_interactions"]
    want_forces = bool(spec.get("forces", True))
    padded = S.Rij in data

    def evaluate(x):
        if padded:
            x = model.representation(x)
            return model.output_modules[0](x)
        return model(x)

    resident = batch_to_device(data, dev)

    def fresh(x):
        # the model writes into the dict and sets requires_grad on positions: hand it a shallow copy each step
        y = dict(x)
        ops._GRAPH_CACHE.clear()  # every step rebuilds the CSR/sender views from idx_i/idx_j (no cached work)
        if S.R in y:
            y[S.R] = y[S.R].detach()
        return y

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def flush_l2():
        flush_buf.fill_(1)

    # ---- per-kernel live timing of the fused edge kernels (CUDA events on the launch stream) -------------------
    # With the CUDA-graph path the events are "external" events: recorded inside the capture they become event-record
    # nodes of the graph, so every replay of the timed region re-records them around the edge-kernel nodes.
    from schnetpack_b200.model import GraphedPotential

    use_graph = not (padded or args.no_graph)
    ev = {"fwd": [], "bwd": []}
    orig_fwd, orig_bwd = ops.painn_edge_fwd, ops.painn_edge_bwd
    timing = {"on": False}

    def new_event():
        return torch.cuda.Event(enable_timing=True, external=True) if use_graph else torch.cuda.Event(True)

    def timed_fwd(x, mu, *a, **k):
        if not timing["on"]:
            return orig_fwd(x, mu, *a, **k)
        s, e = new_event(), new_event()
        s.record()
        r = orig_fwd(x, mu, *a, **k)
        e.record()
        ev["fwd"].append((s, e, mu is not None))
        return r

    def timed_bwd(x, mu, *a, **k):
        if not timing["on"]:
            return orig_bwd(x, mu, *a, **k)
        s, e = new_event(), new_event()
        s.record()
        r = orig_bwd(x, mu, *a, **k)
        e.record()
        ev["bwd"].append((s, e, mu is not None))
        return r

    ops.painn_edge_fwd, ops.painn_edge_bwd = timed_fwd, timed_bwd
    cf_ev = []                                   # (start, end, graph) per timed launch of the fused SchNet block kernel
    orig_cf = ops.schnet_cfconv_fwd_tc

    def timed_cf(h, phi, geo, graph, *a, **k):
        if not timing["on"]:
            return orig_cf(h, phi, geo, graph, *a, **k)
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record()
        r = orig_cf(h, phi, geo, graph, *a, **k)
        e.record()
        cf_ev.append((s, e, graph.rowptr[graph.n_atoms:]))     # only the device count of active edges, not the graph
        return r

    ops.schnet_cfconv_fwd_tc = timed_cf

    # ---- device-resident timing -----------------------------------------------------------------------------------
    # One step = one E+F evaluation of the resident batch, graph-view build included.  Default: replay of the captured
    # evaluation (GraphedPotential, the product's steady-state path -- the eager Python loop is launch-bound on the host
    # at this kernel granularity); --no-graph times eager model(inputs) calls instead.
    kernel_ms = {"fwd": [], "bwd": []}          # (ms, has_mu) per timed edge-kernel launch
    evaluate(fresh(resident))                   # one-time work (weight packing, kernel attributes) outside the counts
    torch.cuda.synchronize()
    timing["on"] = spec["kind"] == "painn" or not use_graph
    if use_graph:
        g_res = GraphedPotential(model)
        c0 = _lib.launch_count
        g_res(resident)                          # 2 eager warm-ups + capture
        launches_per_step = (_lib.launch_count - c0) // (g_res.warmup + 1)
        n_bwd = len(ev["bwd"]) // (g_res.warmup + 1)
        n_fwd = len(ev["fwd"]) // (g_res.warmup + 1)
        pairs = {"fwd": ev["fwd"][-n_fwd:] if n_fwd else [], "bwd": ev["bwd"][-n_bwd:] if n_bwd else []}

        def step():
            return g_res.replay()
    else:
        launches_per_step = None
        pairs = None

        def step():
            return evaluate(fresh(resident))

    sampler = ClockSampler(local_rank) if rank == 0 else None   # polls every 100 ms from the warm-up on (GPU under load)
    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    ev["fwd"].clear()
    ev["bwd"].clear()
    cf_ev.clear()
    if dist is not None:
        dist.barrier()
    launches0 = _lib.launch_count
    step_ev = []
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.mark()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush_l2()
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record()
        out = step()
        e.record()
        step_ev.append((s, e))
        if use_graph:                           # the external events are re-recorded by every replay: read them now
            torch.cuda.synchronize()
            for kind in ("fwd", "bwd"):
                kernel_ms[kind] += [(a.elapsed_time(b), hm) for a, b, hm in pairs[kind]]
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: out[k].detach().cpu().numpy() for k in model.model_outputs if k in out})
    launches = launches_per_step * args.steps if use_graph else _lib.launch_count - launches0
    timing["on"] = False
    if not use_graph:
        for kind in ("fwd", "bwd"):
            kernel_ms[kind] = [(a.elapsed_time(b), hm) for a, b, hm in ev[kind]]
    clocks = sampler.stop() if sampler is not None else None
    dev_ms = sum(s.elapsed_time(e) for s, e in step_ev)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)

    # ---- end-to-end: pinned host buffers -> H2D -> model -> D2H(energy, forces) -------------------------------------
    host = {}
    for k, v in data.items():
        tt = torch.as_tensor(v)
        if tt.is_floating_point():
            tt = tt.float()
        host[k] = tt.pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    e_host = torch.empty(B, dtype=torch.float32).pin_memory()
    f_host = torch.empty((N, 3), dtype=torch.float32).pin_memory() if want_forces else None
    d2h = e_host.numel() * 4 + (f_host.numel() * 4 if f_host is not None else 0)

    graphed = GraphedPotential(model) if use_graph else None

    def e2e_step():
        # public API call a user makes: host batch in, energy/forces out.  GraphedPotential copies the pinned host
        # tensors into its static device buffers (H2D, non-blocking) and replays the captured evaluation.
        if graphed is not None:
            o = graphed(host)
        else:
            x = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
            o = evaluate(x)
        e_host.copy_(o["energy"], non_blocking=True)
        if f_host is not None:
            f_host.copy_(o["forces"], non_blocking=True)

    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e2e_ev = []
    for _ in range(args.steps):
        flush_l2()
        s, e = torch.cuda.Event(True), torch.cuda.Event(True)
        s.record()
        e2e_step()
        e.record()
        e2e_ev.append((s, e))
    torch.cuda.synchronize()
    t2 = torch.tensor([sum(s.elapsed_time(e) for s, e in e2e_ev)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.barrier()
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t2.item()) * 1e-3)
    e2e_steps_ms = sorted(s.elapsed_time(e) for s, e in e2e_ev)

    if rank != 0:
        return

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------------
    peak, peak_src = measured_peaks()
    roof = None
    roof_all = {}
    if kernel_ms["fwd"] or kernel_ms["bwd"]:
        for kind in ("fwd", "bwd"):
            if not kernel_ms[kind]:
                continue
            tot_ms = sum(ms for ms, _ in kernel_ms[kind])
            tot_bytes = sum(edge_kernel_bytes(E, N, F, hm, kind == "bwd") for _, hm in kernel_ms[kind])
            n = len(kernel_ms[kind])
            ach = tot_bytes / (tot_ms * 1e-3) / 1e9
            roof_all[kind] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                              "traffic": None,
                              "kernel": f"k_painn_edge_{kind}" + ("_tc" if ops.edge_tc_ok(F, spec.get("n_rbf", 20), E) else ""),
                              "launches_timed": n,
                              "avg_us": 1e3 * tot_ms / n, "algorithmic_bytes_per_launch": tot_bytes / n,
                              "share_of_step": tot_ms / dev_ms, "peak_source": peak_src,
                              "model": "algorithmic bytes = no-reuse gather model of SURVEY 8(d): every gathered row counted as "
                                       "HBM traffic; rows served by the 126 MB L2 let frac approach or exceed 1 -- `traffic` is "
                                       "the DRAM bytes ncu measured",
                              "timing": "CUDA events around the kernel, inside the timed region"
                                        + (" (external event nodes of the replayed graph)" if use_graph else "")}
        dom = max(roof_all, key=lambda k: roof_all[k]["share_of_step"])
        roof = dict(roof_all[dom])
        tr = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tr) and args.config == "cfg2" and args.batch in (None, 256):   # the ncu capture is of this workload
            try:
                roof["traffic"] = json.load(open(tr)).get(roof["kernel"])
            except Exception:
                pass

    if cf_ev:      # fused SchNet block kernel: tensor-pipe bound (SURVEY 8d: 2(R F + F^2) = 37.9 kFLOP per edge and layer)
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
        tpeak = float(d.get("bf16_tflops", 1750.0))
        n_act = int(cf_ev[0][2][0])
        ms_l = [a.elapsed_time(b) for a, b, _ in cf_ev]
        flops = n_act * 2.0 * (spec.get("n_rbf", 20) * F + F * F)
        ach = flops * len(ms_l) / (sum(ms_l) * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": None,
                "kernel": "k_schnet_cfconv_fwd_tc", "launches_timed": len(ms_l), "avg_us": 1e3 * sum(ms_l) / len(ms_l),
                "active_edges": n_act, "edge_slots": E, "share_of_step": sum(ms_l) / dev_ms,
                "peak_source": "MEASURED_PEAKS.json bf16 dense burst" if d else "fallback (B200_PROFILING.md)",
                "model": "algorithmic fp32 FLOPs of the filter network over the ACTIVE edges (padding slots dropped); the kernel "
                         "computes in 3xTF32 (3 MMAs per product, TF32 = 1/2 of the bf16 rate): its own ceiling is peak / 6",
                "timing": "CUDA events around the kernel, inside the timed region"}
        roof_all = {"cfconv_fwd": roof}

    # ---- CPU baseline (bounded sample, rank 0, N=1 only): the reference's own modules when oracle/_ref is present ----------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_leg(args)

    # ---- the reference's eager single-GPU path (its own modules .to(cuda)) on this B200, for the >=5x target ---------------
    eager = None
    if world == 1 and not args.no_cpu_baseline:
        eager = eager_gpu_leg(spec, params, data, dev, B)

    md_info = None
    if args.md and world == 1 and S.cell in data and not padded:
        # device-resident MD step (row f1 + f2): velocity Verlet + neighbour list rebuilt on the device + E/F, one CUDA graph
        from schnetpack_b200.md import DeviceMD
        from schnetpack_b200.neighbors import neighbor_list

        masses = torch.ones(N, device=dev)
        md = DeviceMD(model, resident, masses, time_step=1e-4, cutoff=spec["cutoff"], capacity=int(E * 1.15))
        md.run(5)
        torch.cuda.synchronize()
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        md.run(50)
        e_.record()
        torch.cuda.synchronize()
        md_ms = s_.elapsed_time(e_) / 50
        nat = resident[S.n_atoms]
        for _ in range(3):
            neighbor_list(resident[S.R], resident.get(S.cell), resident.get(S.pbc), nat, spec["cutoff"], capacity=int(E * 1.15), pad=True)
        torch.cuda.synchronize()
        s_.record()
        for _ in range(20):
            neighbor_list(resident[S.R], resident.get(S.cell), resident.get(S.pbc), nat, spec["cutoff"], capacity=int(E * 1.15), pad=True)
        e_.record()
        torch.cuda.synchronize()
        md_info = {"ms_per_md_step": md_ms, "neighbor_list_ms": s_.elapsed_time(e_) / 20, "capacity": int(E * 1.15),
                   "pairs": int(md.n_pairs[0]), "overflow": int(md.n_pairs[1]),
                   "what": "velocity Verlet + device cell-list rebuild (every step, no skin) + E/F, CUDA-graph replay"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": config_dict(args, world, B, N, E, F, T),
        "step": ("CUDA-graph replay of model(inputs) on the resident batch (GraphedPotential.replay)" if use_graph
                 else "eager model(inputs) on the resident batch"),
        "edge_msgs_per_s": world * E * T * args.steps / (total_ms * 1e-3),
        "wall_ms_per_step": 1e3 * t_wall / args.steps,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "eager model(inputs)" if graphed is None else "GraphedPotential(model)(host_batch): CUDA-graph replay",
                "ms_per_step_median": e2e_steps_ms[len(e2e_steps_ms) // 2], "ms_per_step_max": e2e_steps_ms[-1]},
        "gpu_launches": launches,
        "roofline": roof, "roofline_all": roof_all, "cpu_baseline": cpu, "eager_gpu_baseline": eager,
        "vs_reference_gpu_eager": (value / eager["value"] if eager and "value" in eager else None),
        "e2e_vs_reference_gpu_eager": (e2e_value / eager["value"] if eager and "value" in eager else None),
        "impl_switches": {"dense": ops.DENSE_IMPL, "edge": ops.EDGE_IMPL, "chain": ops.CHAIN_IMPL, "cfconv": ops.CFCONV_IMPL},
    }
    ops.painn_edge_fwd, ops.painn_edge_bwd, ops.schnet_cfconv_fwd_tc = orig_fwd, orig_bwd, orig_cf
    if md_info is not None:
        line["md"] = md_info
    return line


# ------------------------------------------------------------------------------------------------- spatial (cfg5) arm
def run_spatial(args, rank, world, local_rank, steps=None, warmup=None, cpu_leg=True, dump_dir=None):
    """cfg5: ONE periodic box (default 262144 atoms, PaiNN 128x3, E+F) cut into `world` slabs; every rank owns a slab, holds
    read-only ghost rows of the senders it does not own, and exchanges (x, mu) ghost rows per interaction block over NCCL
    point-to-point (gradients back in the reverse sweep).  STRONG scaling: the box is fixed, `value` = whole-box evaluations
    per second.  At N=1 the same pipeline runs without a halo -- the single-GPU workload whose gathered tables (400 MB per
    [N,3F] table) exceed the 126 MB L2, where the roofline fraction of the edge kernels is an HBM statement."""
    from schnetpack_b200 import _lib, ops, parallel as P
    from schnetpack_b200.model import from_spec
    from schnetpack_b200.neighbors import neighbor_list

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=dev)
    steps = steps or args.steps
    warmup = args.warmup if warmup is None else warmup
    n_total = args.atoms or 262144
    spec = S.model_spec(**S.CONFIGS["cfg5"]["spec"])
    box = S.periodic_box(n_total, build_list=False)
    params = S.init_params(spec, seed=0)
    model = from_spec(spec, params, dev)
    F, T = spec["n_atom_basis"], spec["n_interactions"]
    # the neighbour list of the whole box, built on the device (linked-cell kernel), then the graph partition on the host
    R_all = torch.as_tensor(box[S.R], device=dev)
    ii, jj, off, _ = neighbor_list(R_all, torch.as_tensor(box[S.cell], device=dev), torch.as_tensor(box[S.pbc], device=dev),
                                   torch.as_tensor(box[S.n_atoms], device=dev), spec["cutoff"])
    box[S.idx_i], box[S.idx_j], box[S.offsets] = ii.cpu().numpy(), jj.cpu().numpy(), off.cpu().numpy()
    E_total = int(box[S.idx_i].shape[0])
    del ii, jj, off, R_all
    torch.cuda.empty_cache()
    owner = P.slab_owners(box[S.R], world)
    plan = P.partition_graph(owner, box[S.idx_i], box[S.idx_j], rank, world)
    engine = P.PartitionedPotential(model, box, plan, dev, group=None)
    E_loc, N_loc = int(plan.idx_i.shape[0]), plan.n_owned + plan.n_ghost
    halo_rows = plan.n_ghost
    box.pop(S.idx_i), box.pop(S.idx_j), box.pop(S.offsets)

    # ---- live timing of the edge kernels (CUDA events on the launch stream, inside the timed region)
    ev = {"fwd": [], "bwd": []}
    orig_fwd, orig_bwd = ops.painn_edge_fwd, ops.painn_edge_bwd
    timing = {"on": False}

    def timed(kind, orig):
        def f(x, mu, *a, **k):
            if not timing["on"]:
                return orig(x, mu, *a, **k)
            s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
            s_.record()
            r = orig(x, mu, *a, **k)
            e_.record()
            ev[kind].append((s_, e_, mu is not None))
            return r
        return f

    ops.painn_edge_fwd, ops.painn_edge_bwd = timed("fwd", orig_fwd), timed("bwd", orig_bwd)
    # halo share: events around every exchange (forward and reverse) on the launch stream
    halo_ev = []
    orig_halo_f, orig_halo_b = P.HaloExchange.forward, P.HaloExchange.backward

    def halo_f(ctx, rows, plan_, group=None):
        if not timing["on"]:
            return orig_halo_f(ctx, rows, plan_, group)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        r = orig_halo_f(ctx, rows, plan_, group)
        e_.record()
        halo_ev.append((s_, e_))
        return r

    def halo_b(ctx, g):
        if not timing["on"]:
            return orig_halo_b(ctx, g)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        r = orig_halo_b(ctx, g)
        e_.record()
        halo_ev.append((s_, e_))
        return r

    P.HaloExchange.forward, P.HaloExchange.backward = staticmethod(halo_f), staticmethod(halo_b)
    orig_peer_f, orig_peer_b = P.PeerHaloExchange.forward, P.PeerHaloExchange.backward

    def peer_f(ctx, rows, halo):
        if not timing["on"]:
            return orig_peer_f(ctx, rows, halo)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        r = orig_peer_f(ctx, rows, halo)
        e_.record()
        halo_ev.append((s_, e_))
        return r

    def peer_b(ctx, g):
        if not timing["on"]:
            return orig_peer_b(ctx, g)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        r = orig_peer_b(ctx, g)
        e_.record()
        halo_ev.append((s_, e_))
        return r

    P.PeerHaloExchange.forward, P.PeerHaloExchange.backward = staticmethod(peer_f), staticmethod(peer_b)

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(warmup, 3)):
        energy, forces = engine()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    timing["on"] = True
    c0 = _lib.launch_count
    step_ev = []
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.mark()
    for _ in range(steps):
        flush_buf.fill_(1)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        energy, forces = engine()
        e_.record()
        step_ev.append((s_, e_))
    torch.cuda.synchronize()
    timing["on"] = False
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"energy": energy.detach().cpu().numpy(), "forces": forces.detach().cpu().numpy()})
    launches = _lib.launch_count - c0
    clocks = sampler.stop() if sampler is not None else None
    dev_ms = sum(a.elapsed_time(b) for a, b in step_ev)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    halo_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in halo_ev)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(halo_ms, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / steps
    value = steps / (total_ms * 1e-3)                      # whole-box evaluations per second (all ranks together)

    # ---- end to end: host positions in, energy + owned forces out
    R_host = engine.R_own.detach().cpu().pin_memory()
    f_host = torch.empty((plan.n_owned, 3), dtype=torch.float32).pin_memory()
    e_host = torch.empty(1, dtype=torch.float32).pin_memory()
    h2d, d2h = R_host.numel() * 4, f_host.numel() * 4 + 4

    def e2e_step():
        engine.set_positions(R_host.to(dev, non_blocking=True))
        e_, f_ = engine()
        e_host.copy_(e_, non_blocking=True)
        f_host.copy_(f_, non_blocking=True)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    e2e_ev = []
    for _ in range(steps):
        flush_buf.fill_(1)
        s_, e_ = torch.cuda.Event(True), torch.cuda.Event(True)
        s_.record()
        e2e_step()
        e_.record()
        e2e_ev.append((s_, e_))
    torch.cuda.synchronize()
    t2 = torch.tensor([sum(a.elapsed_time(b) for a, b in e2e_ev)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.barrier()
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = steps / (float(t2.item()) * 1e-3)
    ops.painn_edge_fwd, ops.painn_edge_bwd = orig_fwd, orig_bwd
    P.HaloExchange.forward, P.HaloExchange.backward = staticmethod(orig_halo_f), staticmethod(orig_halo_b)
    P.PeerHaloExchange.forward, P.PeerHaloExchange.backward = staticmethod(orig_peer_f), staticmethod(orig_peer_b)
    transport = engine.transport
    del engine
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peak, peak_src = measured_peaks()
    roof_all = {}
    for kind in ("fwd", "bwd"):
        if not ev[kind]:
            continue
        ms_l = [(a.elapsed_time(b), hm) for a, b, hm in ev[kind]]
        tot_ms = sum(m for m, _ in ms_l)
        tot_bytes = sum(edge_kernel_bytes(E_loc, N_loc, F, hm, kind == "bwd") for _, hm in ms_l)
        ach = tot_bytes / (tot_ms * 1e-3) / 1e9
        roof_all[kind] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                          "kernel": f"k_painn_edge_{kind}_tc", "launches_timed": len(ms_l), "avg_us": 1e3 * tot_ms / len(ms_l),
                          "algorithmic_bytes_per_launch": tot_bytes / len(ms_l), "share_of_step": tot_ms / dev_ms,
                          "peak_source": peak_src,
                          "model": "SURVEY 8(d) no-reuse gather model over this rank's edges / local rows; the gathered "
                                   "tables (N_local x 1.5 KB x 2) exceed the 126 MB L2 here",
                          "timing": "CUDA events around the kernel, inside the timed region (rank 0)"}
    roof = None
    if roof_all:
        dom = max(roof_all, key=lambda k: roof_all[k]["share_of_step"])
        roof = dict(roof_all[dom])
        tr = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tr):
            try:
                roof["traffic"] = json.load(open(tr)).get(f"cfg5_n{world}_" + roof["kernel"])
            except Exception:
                pass
    cpu = None
    if world == 1 and not args.no_cpu_baseline and cpu_leg:
        cpu = cpu_baseline_leg(args)
    line = {
        "metric": METRIC, "value": value, "unit": "box-evals/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": config_dict(args, world, 1, n_total, E_total, F, T),
        "step": "eager per-block pipeline (context net -> halo exchange -> fused edge kernel -> mixing) + autograd reverse sweep",
        "edge_msgs_per_s": E_total * T * steps / (total_ms * 1e-3),
        "atoms_per_s": n_total * steps / (total_ms * 1e-3),
        "rank0": {"owned_atoms": plan.n_owned, "ghost_atoms": halo_rows, "local_edges": E_loc},
        "halo": {"exchanges_per_step": len(halo_ev) // max(steps, 1), "ms_per_step_max_over_ranks": float(halo_ms.item()) / steps,
                 "share_of_step": float(halo_ms.item()) / total_ms,
                 # forward: positions (3) + x (3F) per block + mu (3F) from the second block on; the reverse sweep sends the
                 # same volume back (gradients of the ghost rows to their owners)
                 "bytes_sent_per_step_rank0": 2 * 4 * int(sum(len(v) for v in plan.send.values())) * (3 + 3 * F * T + 3 * F * (T - 1)),
                 "transport": {"peer": "NVLink peer memory: spk_halo_pull / spk_halo_pull_add over torch symmetric memory, one device-side barrier per exchange",
                               "p2p": "NCCL grouped isend/irecv (torch.distributed.batch_isend_irecv), index-gather pack, receives land in the ghost block",
                               "none": "single rank"}[transport]},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "box-evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "PartitionedPotential.set_positions(host) -> __call__() -> energy, forces to pinned host"},
        "gpu_launches": launches,
        "roofline": roof, "roofline_all": roof_all, "cpu_baseline": cpu,
        "impl_switches": {"dense": ops.DENSE_IMPL, "edge": ops.EDGE_IMPL},
    }
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(S.CONFIGS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--atoms", type=int, default=None, help="cfg5: atoms in the periodic box (default 262144)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spatial", action="store_true", help="skip the cfg5 strong-scaling leg appended to the default run")
    ap.add_argument("--spatial-steps", type=int, default=8)
    ap.add_argument("--md", action="store_true", help="also time the device-resident MD step (rows f1+f2); not part of the metric")
    ap.add_argument("--no-graph", action="store_true", help="time eager model(inputs) calls (value and e2e) instead of CUDA-graph replays")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0; cfg5: its owned atoms) as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    # the contract is ONE JSON line on stdout: libraries (NCCL's version banner, symmetric-memory set-up) write to fd 1, so
    # everything but the final line is diverted to stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if args.config == "cfg5":
        line = run_spatial(args, rank, world, local_rank, dump_dir=args.dump_outputs)
    else:
        line = run_cuda(args, rank, world, local_rank)
        if not args.no_spatial:
            # second leg, same run: STRONG scaling of the one-box workload (cfg5) on the same N GPUs, so that a 1/2/4/8-GPU
            # sweep of the default command also yields a curve with a real collective (the halo) in the data path
            try:
                sp = run_spatial(args, rank, world, local_rank, steps=args.spatial_steps, warmup=3, cpu_leg=False)
            except Exception as exc:  # pragma: no cover
                sp = {"error": repr(exc)[:300]}
            if line is not None:
                line["spatial"] = sp
    sys.stdout.flush()
    if line is not None:
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        import torch.distributed as dist

        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
