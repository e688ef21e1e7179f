#!/usr/bin/env python
"""bench.py -- refined samples / second of the collaborative-sampling hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--sweep]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic proposals: K_refine refinement steps through
G-tail + D (sampling/collaborator.py:41-88) followed by the MH-GAN accept-reject pass (sampling/idpsampler.py) on
the refined batch.  Default workload = the north_star target: DCGAN-64 (CelebA shape) nets, refine at generator
layer 1 ([4,4,512] map), batch 1024 per GPU, K_refine = 50, momentum, rate 0.1 (BASELINE.json configs[3], layer 1 of
the sweep, at the per-GPU batch of its 8-GPU sharding).  MNIST (configs[1]) and the 2-D config (configs[0]) are
measured beside it under `also`.  With N > 1 (torchrun) every rank refines its own shard (weak scaling); NCCL only
gathers scores / accepted rows / statistics and the accept stage keeps its counts on the device.

Prints ONE JSON line (rank 0).  `value` is device-timed with inputs resident in HBM; `e2e` goes through the public
drop-in API with pinned HOST inputs and host outputs; `roofline` covers every conv / deconv / fc pass of one
refinement step (tcgen05 passes and image-edge passes, time-weighted), each pass timed live with CUDA events;
`cpu_baseline` is the CPU oracle port of the same path timed on this box (N = 1 only).
`--sweep` runs BASELINE configs C3 / C4 / C5 at this world size and writes gpurun_out/sweep_N<world>.json.
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
PKG = os.path.join(ROOT, "collaborative-gan-sampling_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "refined_samples_per_sec"
UNIT = "samples/s"
DEFAULT_WORKLOAD = "dcgan64_l1"

WORKLOADS = {
    # name: (arch, batch per GPU, refine steps, method, rate, weight gain)
    "mnist": ("mnist", 1024, 50, "momentum", 0.1, 3.0),
    "dcgan32_l1": ("dcgan32_l1", 1024, 50, "momentum", 0.1, 2.5),
    "dcgan64_l1": ("dcgan64_l1", 1024, 50, "momentum", 0.1, 2.5),
    "dcgan64_l2": ("dcgan64_l2", 1024, 50, "momentum", 0.1, 2.5),
    "dcgan64_l3": ("dcgan64_l3", 1024, 50, "momentum", 0.1, 2.5),
    "dcgan64_l4": ("dcgan64_l4", 1024, 50, "momentum", 0.1, 2.5),
}
MAX_ROWS_PER_LAUNCH = 8192        # sweep: larger per-GPU batches are refined in chunks of this many rows


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override batch per GPU")
    ap.add_argument("--refine-steps", type=int, default=0, help="override K_refine")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--math", default="tf32", choices=["tf32", "fp32"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements (`also`) in the JSON line")
    ap.add_argument("--no-graph", action="store_true", help="launch the K-step sequence eagerly instead of replaying a CUDA graph")
    ap.add_argument("--sweep", action="store_true", help="BASELINE configs C3/C4/C5 at this world size -> gpurun_out/sweep_N<world>.json")
    ap.add_argument("--sweep-max-seconds", type=float, default=60.0, help="skip sweep points whose estimated step time exceeds this")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as "
                    "DIR/<name>.npy (float32 / float64, at most 60 MiB in all) to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.sweep):
        ap.error("--dump-outputs applies to the timed hot path of --impl ours (not --sweep)")
    return args


DUMP_BYTES = 60 << 20           # under 64 MB in all, .npy headers included


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy, at most DUMP_BYTES in all.  Arrays are written smallest first; one
    larger than an equal share of the bytes still free keeps a fixed, seeded sample of its rows (sorted), so two runs
    with the same arguments write the same rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    free, left = DUMP_BYTES, len(arrays)
    for name in sorted(arrays, key=lambda k: arrays[k].nbytes):
        a = arrays[name]
        share = free // left
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.RandomState(0).choice(a.shape[0], keep, replace=False))]
            print("bench: %s.npy holds a seeded sample of %d of its %d rows" % (name, keep, arrays[name].shape[0]),
                  file=sys.stderr)
        np.save(os.path.join(out_dir, name + ".npy"), a)
        free, left = free - a.nbytes, left - 1


# ----------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks line")
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None             # wall-clock window of the timed region (mark_start / mark_end)

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # samples taken inside the timed window (the sampler starts before the warm-up so it is already running);
        # a window shorter than the sampling period falls back to every sample taken under load
        rows = [r for t, r in self.rows if self.t0 is not None and self.t1 is not None and self.t0 <= t <= self.t1 + 0.05]
        in_window = len(rows)
        if not rows:
            rows = [r for _, r in self.rows]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        # median over the upper half = clocks under load (idle samples before/after the region are low)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_region": in_window}


def measured_peaks():
    """(hbm GB/s, bf16 burst TFLOP/s, bf16 sustained TFLOP/s, source) from the driver-written MEASURED_PEAKS.json, else the
    fallback B200_PROFILING.md states."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), float(j["bf16_tflops"]), float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), \
            "MEASURED_PEAKS.json"
    return 6650.0, 1590.0, 1400.0, "fallback (B200_PROFILING.md: 6.65 TB/s, 1.59 PFLOP/s bf16 burst)"


# ----------------------------------------------------------------------------------------------------------
# CPU oracle port (cpu_baseline / --impl reference)
# ----------------------------------------------------------------------------------------------------------
def host_threads():
    """All host threads this process may use (torchrun pins OMP_NUM_THREADS=1; the CPU arm undoes that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_sample_rows(arch_name, ksteps):
    """Rows of one CPU step: a BOUNDED sample of the workload, about 0.5 TFLOP of algorithmic work (seconds on a
    multi-core host), never more than the reference's default batch of 64 (nsgan/main.py:32)."""
    from oracle import nets as onets            # (the CPU arm never touches the product package or libcgs.so)
    macs = 0.0
    arch = onets.get_arch(arch_name)
    for l in arch["gtail"] + arch["d"]:
        if l["type"] == "fc":
            macs += l["cin"] * l["cout"]
        elif l["type"] == "conv":
            macs += ((l["hin"] + 1) // 2) * ((l["win"] + 1) // 2) * l["cin"] * l["cout"] * l["k"] ** 2
        else:
            macs += l["hin"] * 2 * l["win"] * 2 * l["cin"] * l["cout"] * l["k"] ** 2 / 4.0
    per = 2.0 * (2 * ksteps + 1) * macs
    return int(max(4, min(64, round(0.5e12 / per))))


def cpu_port_step(arch_name, gain, batch, refine_steps, method, rate, seed=0):
    """One hot-path pass on the host: oracle graph refiner (FP32 torch-CPU restatement of
    sampling/collaborator.py over the nsgan nets, D BN in inference mode) + oracle MH chain.  Returns seconds."""
    import numpy as np
    import torch
    from oracle import graph_refiner as gr
    from oracle import nets as onets
    from oracle import sampling_np as snp
    if torch.get_num_threads() != host_threads():
        torch.set_num_threads(host_threads())
    arch = onets.get_arch(arch_name)
    w = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=2019), gain)
    w = {k: torch.from_numpy(v) for k, v in w.items()}
    rng = np.random.RandomState(seed)
    h0 = torch.from_numpy(np.maximum(rng.standard_normal((batch,) + tuple(arch["feature_shape"])), 0).astype(np.float32))
    t0 = time.perf_counter()
    out = gr.build_refiner(h0, arch, w, refine_steps, rate, method=method)
    sig = torch.sigmoid(out["optimal_logit"]).numpy().reshape(-1, 1)
    emit, _, _, _ = snp.mh_chain(sig, rng.rand(batch), np.float32(0.5), 1, 20, 0)
    _ = out["refined"].numpy()[emit] if len(emit) else None
    return time.perf_counter() - t0


def run_reference(args, wl):
    import torch
    arch_name, batch, ksteps, method, rate, gain = wl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_b = cpu_sample_rows(arch_name, ksteps)
    for _ in range(max(args.warmup, 0) and 1):
        cpu_port_step(arch_name, gain, sample_b, ksteps, method, rate)
    times = [cpu_port_step(arch_name, gain, sample_b, ksteps, method, rate, seed=i) for i in range(args.steps)]
    total = sum(times)
    value = sample_b * args.steps / total
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s: refine K=%d %s rate %.2g + MH(T=20)" % (arch_name, ksteps, method, rate),
                   "batch_per_step": sample_b, "note": "CPU oracle port of the reference path (TF 1.13 is not installable); "
                   "each step is a bounded %d-row sample of the %d-row workload (per-row CPU cost is flat in the batch)"
                   % (sample_b, batch)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d steps x %d rows, K=%d" % (args.steps, sample_b, ksteps)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# ours
# ----------------------------------------------------------------------------------------------------------
def measure_tf32_peak(torch, dev):
    """cuBLAS TF32 GEMM 8192^3, best of 5 (burst) -- measured beside the assumed 0.5 x BF16 denominator."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(2):
            a @ b
        best = 1e9
        for _ in range(5):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            a @ b
            e.record()
            e.synchronize()
            best = min(best, s.elapsed_time(e))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def roofline_profile(torch, spec, arch, batch, math, dev, reps=3):
    """Time every conv / deconv / fc pass of one refinement step (forward chain + data-gradient chain) with CUDA
    events on the launching stream, at the benchmark batch size.  Returns per-pass rows."""
    import ctypes as C
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    lib = L.load()
    chain = [(l, spec.gtail.layer_desc(i)) for i, l in enumerate(arch["gtail"])] + \
            [(l, spec.d.layer_desc(i)) for i, l in enumerate(arch["d"][:-1])]
    rows = []
    for layer, desc in chain:
        cin, cout = layer["cin"], layer["cout"]
        if layer["type"] == "fc":
            xs, ys = (batch, cin), (batch, N.cstride(cout))
        elif layer["type"] == "conv":
            xs = (batch, layer["hin"], layer["win"], N.cstride(cin))
            ys = (batch, (layer["hin"] + 1) // 2, (layer["win"] + 1) // 2, N.cstride(cout))
        else:
            xs = (batch, layer["hin"], layer["win"], N.cstride(cin))
            ys = (batch, layer["hin"] * 2, layer["win"] * 2, N.cstride(cout))
        x = torch.randn(xs, device=dev)
        y = torch.empty(ys, device=dev)
        dy = torch.randn(ys, device=dev)
        dx = torch.empty(xs, device=dev)
        ws = torch.empty(int(lib.cgs_layer_workspace_bytes(C.byref(desc), batch)), dtype=torch.uint8, device=dev)
        flops = 2.0 * S.layer_macs(layer) * batch
        for name, fn in (("fwd", lambda: lib.cgs_layer_forward(C.byref(desc), L.MATH_IDS[math], batch, L.ptr(x), L.ptr(y), L.ptr(ws), ws.numel(), L.stream_ptr())),
                         ("bwd", lambda: lib.cgs_layer_backward(C.byref(desc), L.MATH_IDS[math], batch, L.ptr(dy), L.ptr(dx), L.ptr(x), 1, L.ptr(ws), ws.numel(), L.stream_ptr()))):
            L.check(fn())
            best = 1e9
            inner = 10                       # back-to-back launches per event pair: hides the host launch latency
            for _ in range(reps):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(inner):
                    fn()
                e.record()
                e.synchronize()
                best = min(best, s.elapsed_time(e) * 1e-3 / inner)
            # which kernel runs the pass: 0 = tcgen05 gathered GEMM; 1 / 2 = image-edge streaming kernels
            layout = int(lib.cgs_pass_layout(C.byref(desc), 1 if name == "bwd" else 0))
            row = {"layer": layer["name"] + "." + name, "us": round(best * 1e6, 1), "tflops": round(flops / best / 1e12, 1),
                   "kernel": ("conv_gemm_tc", "edge_narrow", "edge_wide")[layout], "flops": flops, "s": best}
            if layout:                        # HBM-bound passes: algorithmic bytes = every operand read / written once
                big = (y if cout > cin else x).numel() * 4        # the 64-channel side, read or written once
                img = (x if cout > cin else y).numel() * 4        # the image side
                aux = (big if layout == 2 else img) if name == "bwd" else 0   # derivative operand of the backward pass
                row["bytes"] = int(big + img + aux)
                row["gbs"] = round((big + img + aux) / best / 1e9, 1)
            rows.append(row)
    return rows


def static_traffic(arch_name, batch):
    """ncu DRAM traffic / tensor-pipe activity of the same launch set, captured ONCE per round and committed
    (profiles/round2_traffic.json): static data, labelled as such -- a bench run cannot be taken under a profiler."""
    for fname in ("round2_traffic.json", "round1_traffic.json"):
        path = os.path.join(ROOT, "profiles", fname)
        if not os.path.exists(path) or batch != 1024:
            continue
        with open(path) as f:
            tj = json.load(f).get("dcgan64" if arch_name == "dcgan64_l1" else arch_name) or {}
        if tj:
            return tj, "static: profiles/%s (ncu --set full capture of this launch set, not measured in this run)" % fname
    return {}, None


def build_roofline(torch, spec, arch, arch_name, batch, math, dev, ksteps, step_s):
    hbm_peak, bf16_burst, bf16_sus, src = measured_peaks()
    tf32_cublas = measure_tf32_peak(torch, dev)
    rows = roofline_profile(torch, spec, arch, batch, math, dev)
    tc = [r for r in rows if r["kernel"] == "conv_gemm_tc"]
    edge = [r for r in rows if r["kernel"] != "conv_gemm_tc"]
    f_all, t_all = sum(r["flops"] for r in rows), sum(r["s"] for r in rows)
    f_tc, t_tc = sum(r["flops"] for r in tc), sum(r["s"] for r in tc)
    t_edge = sum(r["s"] for r in edge)
    peak = 0.5 * bf16_burst
    tj, tsrc = static_traffic(arch_name, batch)
    traffic = None
    if "conv_gemm_tc" in tj:
        traffic = int(tj["conv_gemm_tc"]["traffic_bytes"]) + int((tj.get("edge") or {}).get("traffic_bytes", 0))
    per_layer = [{k: v for k, v in r.items() if k not in ("flops", "s")} for r in rows]
    roof = {
        "bound": "tensor",
        "kernel": "every conv / deconv / fc pass of one refinement step (forward + data-gradient chain): "
                  "conv_gemm_tc_kernel (tcgen05 kind::tf32) + the image-edge kernels, time-weighted",
        "achieved": round(f_all / t_all / 1e12, 2), "peak": round(peak, 1), "unit": "TFLOP/s",
        "frac": round(f_all / t_all / 1e12 / peak, 4),
        "traffic": traffic, "traffic_source": tsrc,
        "peak_source": "0.5 x %s bf16_tflops burst (TF32 = half the BF16 rate; passes are timed alone, back to back)" % src,
        "cublas_tf32_tflops_same_run": round(tf32_cublas, 1),
        "frac_of_cublas_tf32": round(f_all / t_all / 1e12 / tf32_cublas, 4),
        "algorithmic_gflop_per_launch_set": round(f_all / 1e9, 2),
        "us_per_launch_set": round(t_all * 1e6, 1),
        "step_share_of_conv_time": round(t_all * (2 * ksteps + 1) / 2.0 / step_s, 3),
        "tcgen05": {"achieved": round(f_tc / t_tc / 1e12, 2), "frac": round(f_tc / t_tc / 1e12 / peak, 4),
                    "us": round(t_tc * 1e6, 1), "gflop": round(f_tc / 1e9, 2),
                    "ncu_tensor_pipe_active_pct": (tj.get("conv_gemm_tc") or {}).get("tensor_pipe_active_pct_time_weighted"),
                    "ncu_source": tsrc},
        "per_layer": per_layer,
    }
    if edge:
        b_edge = sum(r["bytes"] for r in edge)
        roof["edge"] = {"bound": "hbm", "kernel": "image-edge passes (tcgen05 resident-patch kernels on the space-to-depth image, csrc/edge_tc.cu; mma.sync streaming kernels of csrc/edge_conv.cu on maps narrower than 16)",
                        "achieved": round(b_edge / t_edge / 1e9, 1), "peak": hbm_peak, "unit": "GB/s",
                        "frac": round(b_edge / t_edge / 1e9 / hbm_peak, 4), "peak_source": src + " hbm_gbs",
                        "algorithmic_bytes_per_launch_set": int(b_edge), "us": round(t_edge * 1e6, 1),
                        "note": "timed through the dense single-layer entry point: the two window passes include a "
                                "layout copy that the refinement chain does not run"}
    return roof


def make_hot_path(torch, D, refiner, mh, world, rank, batch):
    """refine -> global scores -> MH chain -> accepted rows (global order).  No host synchronisation anywhere: the
    accepted-row count stays a device scalar (padded outputs), the multi-GPU merge is one int32 all-reduce."""
    lo, hi = rank * batch, (rank + 1) * batch

    def hot_path(h0):
        x = refiner.build_refiner(h0, None, "deterministic")
        sig_local = torch.sigmoid(refiner.optimal_logit)
        sig = D.gather_scores(sig_local, sizes=[batch] * world) if world > 1 else sig_local
        emit, cnt = mh.select_async(sig)
        if world > 1:
            acc, cnt = D.gather_accepted_async(x, emit, cnt, lo, hi)
        else:
            acc, cnt = mh.gather_async(x)                        # cgs_gather_rows on the emitted source rows
        return x, acc, cnt, sig_local
    return hot_path


def timed_steps(torch, dist, hot_path, h0, steps, warmup, world, flush=None, clocks=None):
    """W warm-up steps, then K timed steps (CUDA events per step on the current stream, L2 flushed in between),
    bracketed by barrier + synchronize; returns (seconds, max over ranks; last outputs)."""
    out = None
    for _ in range(warmup):
        out = hot_path(h0)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if clocks:
        clocks.mark_start()
    step_ms = []
    torch.cuda.synchronize()
    for _ in range(steps):
        if flush is not None:
            flush.fill_(1)                   # flush L2 between timed iterations (outside the event pair)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = hot_path(h0)
        e.record()
        e.synchronize()
        step_ms.append(s.elapsed_time(e))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if clocks:
        clocks.mark_end()
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    return float(total_ms.item()) * 1e-3, out


def measure_extra(torch, name, dev, math, steps, warmup):
    """Device-timed run of another workload (inputs resident, CUDA events, L2 flushed between steps)."""
    from cgs import dist as D
    from cgs import nets as N
    from cgs import synthetic as S
    from sampling.collaborator import Refiner
    from sampling.idpsampler import IndependenceSampler
    import numpy as np
    arch_name, batch, ksteps, method, rate, gain = WORKLOADS[name]
    arch = N.get_arch(arch_name)
    spec = N.NetSpec(arch, S.init_weights(arch, seed=2019, gain=gain), dev, math=math)
    refiner = Refiner(ksteps, rate, method, cuda_graph=True)
    refiner.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    mh = IndependenceSampler(T=20, rng="philox", seed=2019)
    mh.set_score_curr(np.float32(0.5))
    h0 = torch.from_numpy(S.proposal_features(arch, batch, seed=7)).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    hot = make_hot_path(torch, D, refiner, mh, 1, 0, batch)
    t, _ = timed_steps(torch, None, hot, h0, steps, warmup, 1, flush)
    t /= steps
    flops = S.refine_flops_per_sample(arch, ksteps) * batch
    _, bf16_burst, bf16_sus, src = measured_peaks()
    out = {"value": batch / t, "unit": UNIT, "ms_per_step": t * 1e3, "steps": steps, "warmup": warmup,
           "workload": "%s: refine K=%d %s + MH(T=20), batch %d" % (arch_name, ksteps, method, batch),
           "tflops_algorithmic": round(flops / t / 1e12, 1),
           "frac_of_tf32_peak_sustained": round(flops / t / 1e12 / (0.5 * bf16_sus), 3),
           "peak_note": "0.5 x %s bf16_tflops_sustained (whole-step number, kernels timed inside a long step)" % src}
    del refiner, spec, flush
    torch.cuda.empty_cache()
    return out


def measure_early_exit(torch, spec, arch, h0, ksteps, method, rate, dev, steps=3, warmup=2):
    """Opt-in early exit (README.md:13): samples/s against the fraction of the batch that left before step K.
    Thresholds are quantiles of the batch's final best logits; compaction and grid sizing are device-side, the
    K-step sequence is replayed as a CUDA graph exactly like the plain run."""
    from cgs import nets as N
    from sampling.collaborator import Refiner
    base = Refiner(ksteps, rate, method, cuda_graph=True)
    base.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    base.build_refiner(h0)
    logits = base.optimal_logit.float()
    rows = []
    for q in (1.01, 0.75, 0.5, 0.25):
        thr = float(torch.quantile(logits, min(q, 1.0))) + (1e6 if q > 1 else 0.0)
        r = Refiner(ksteps, rate, method, cuda_graph=True)
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        r.early_exit_logit = thr
        for _ in range(warmup):
            r.build_refiner(h0)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            r.build_refiner(h0)
        e.record()
        e.synchronize()
        t = s.elapsed_time(e) * 1e-3 / steps
        exited = float((r.optimal_logit >= thr).float().mean())
        mean_steps = float(torch.where(r.optimal_logit >= thr, r.optimal_step, torch.full_like(r.optimal_step, ksteps)).mean())
        rows.append({"exit_logit": None if q > 1 else round(thr, 4), "fraction_exited": round(exited, 4),
                     "mean_steps_executed": round(mean_steps, 2), "ms_per_step": round(t * 1e3, 3),
                     "samples_per_s": round(h0.shape[0] / t, 1)})
        del r
    del base
    torch.cuda.empty_cache()
    return {"config": {"early_exit": "device-side threshold test + ordered compaction, no host sync, CUDA graph replay"},
            "rows": rows}


def measure_2d(torch, dev, n=10000, steps_k=50, reps=5, cpu=True):
    """BASELINE config 0: imbalanced-8-Gaussians-style 2-D MLP GAN, collaborative refine (ladam, K=50) + DRS + MH on
    N=10 000 points (synthetic/main.py:299).  Device-timed; beside it the oracle port of refiner_cpu on the host."""
    import types
    import numpy as np
    from cgs import synthetic as S
    from sampling.idpsampler import IndependenceSampler
    from sampling.refiner_cpu import MlpSpec, Refiner
    from sampling.rejector import Rejector
    ws = S.init_mlp2d(64, 6, seed=2019, gain=1.5)
    mlp = MlpSpec(ws, dev)
    rng = np.random.RandomState(0)
    x0 = torch.from_numpy((rng.randn(n, 2) * 4).astype(np.float32)).to(dev)
    real = (rng.randn(n, 2) * 3).astype(np.float32)
    real_mean = float(np.mean(mlp.score(real)[0].cpu().numpy()))
    ref = Refiner(types.SimpleNamespace(rollout_steps=steps_k, rollout_rate=0.1, rollout_method="ladam"))
    ref.set_env(mlp, None, None)
    rej = Rejector(rng="philox", seed=1)
    mh = IndependenceSampler(T=20, rng="philox", seed=2)
    mh.set_score_curr(np.float32(real_mean))
    best, best_refine = 1e9, 1e9
    for it in range(reps + 2):
        s, m, e = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        s.record()
        x = ref.manipulate_sample(x0, "deterministic", real_sigmoid_mean=real_mean)
        m.record()
        sig, _ = mlp.score(x)
        rej.sampling(x, sig, shift_percent=100.0)
        mh.sampling(x, sig)
        e.record()
        e.synchronize()
        if it >= 2:
            best = min(best, s.elapsed_time(e) * 1e-3)
            best_refine = min(best_refine, s.elapsed_time(m) * 1e-3)
    # roofline of the fused refinement kernel: SMEM-resident weights, bound by FP32 FMA issue (SURVEY §8d):
    # 148 SMs x 128 FP32 lanes x 2 FLOP x SM clock
    flop_point = 2.0 * ((steps_k + 1) + steps_k) * 16576          # fwd MACs (K+1 evaluations) + bwd MACs (K)
    props = torch.cuda.get_device_properties(dev)
    clk_ghz = props.clock_rate / 1e6 if hasattr(props, "clock_rate") else 1.965
    fma_peak = props.multi_processor_count * 128 * 2 * clk_ghz / 1e3
    out = {"value": n / best, "unit": "refined points/s", "ms_per_pass": best * 1e3,
           "workload": "2-D MLP D (2-64x5-1), N=%d, ladam K=%d, then DRS(p=100) and MH(T=20)" % (n, steps_k),
           "mflop_per_point": round(flop_point / 1e6, 3),
           "roofline": {"bound": "fp32_fma", "kernel": "mlp2d_refine_split_kernel (one launch for all K steps, four threads per point)",
                        "achieved": round(n * flop_point / best_refine / 1e12, 2), "peak": round(fma_peak, 1),
                        "unit": "TFLOP/s", "frac": round(n * flop_point / best_refine / 1e12 / fma_peak, 4),
                        "us": round(best_refine * 1e6, 1),
                        "peak_source": "%d SMs x 128 FP32 lanes x 2 x %.3f GHz (device max clock); weights are "
                                       "shared-memory resident, only x in / x out touch HBM" % (props.multi_processor_count, clk_ghz),
                        "note": "N = 10^4 points is %d point-warps on %d SMs; bound by the shared-memory pipe (warp-broadcast "
                                        "LDS.128 weight reads, 4 FMAs per load: 69 %% of peak wavefronts in ncu, "
                                        "profiles/round2_ncu_summary.md E)" % ((n + 31) // 32, props.multi_processor_count)}}
    if cpu:
        from oracle import nets as onets
        from oracle import sampling_np as snp
        torch.set_num_threads(host_threads())
        x0h = x0.cpu().numpy()
        t0 = time.perf_counter()
        o = snp.refine_2d(x0h, lambda x: onets.mlp2d_sigmoid_saliency(x, ws), np.float32(real_mean), steps_k, 0.1, "ladam")
        sg, _ = onets.mlp2d_sigmoid_saliency(o["optimal_batch"], ws)
        snp.drs_accept(sg, rng.rand(n), 0.0, shift_percent=100.0)
        snp.mh_chain(sg, rng.rand(n), np.float32(real_mean), 1, 20, 0)
        t = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n / t, "unit": "refined points/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": "same N, one pass (reference refiner_cpu algorithm, torch-CPU MLP)"}
    return out


def setup_dist(torch):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200: libcgs has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    return dist, rank, local_rank, world, dev


def run_ours(args, wl):
    import numpy as np
    import torch
    from cgs import dist as D
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    from sampling.collaborator import Refiner
    from sampling.idpsampler import IndependenceSampler

    arch_name, batch, ksteps, method, rate, gain = wl
    dist, rank, local_rank, world, dev = setup_dist(torch)
    lib = L.load()

    arch = N.get_arch(arch_name)
    weights = S.init_weights(arch, seed=2019, gain=gain)
    spec = N.NetSpec(arch, weights, dev, math=args.math)
    refiner = Refiner(ksteps, rate, method, cuda_graph=not args.no_graph)
    refiner.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    mh = IndependenceSampler(T=20, rng="philox", seed=2019)          # nsgan/GAN.py:169
    mh.set_score_curr(np.float32(0.5))
    h0_host = torch.from_numpy(S.proposal_features(arch, batch, seed=1000 + rank)).pin_memory()
    h0_dev = h0_host.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    hot_path = make_hot_path(torch, D, refiner, mh, world, rank, batch)

    # ---- device-timed region: inputs resident in HBM ------------------------------------------------------
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()                       # running through the warm-up; only samples inside the timed window count
    for _ in range(1):
        hot_path(h0_dev)                     # first call captures the CUDA graph (not one of the W warm-up steps)
    launches0 = lib.cgs_launch_count() + refiner.replayed_launches
    total_s, (x, acc, cnt, sig_local) = timed_steps(torch, dist, hot_path, h0_dev, args.steps, args.warmup, world, flush,
                                                    clocks if rank == 0 else None)
    launches = (lib.cgs_launch_count() + refiner.replayed_launches - launches0) // max(args.steps + args.warmup, 1)
    clk = clocks.stop() if rank == 0 else None
    n_acc = int(cnt.item())
    if args.dump_outputs and rank == 0:
        # what a caller of the hot path receives from the last timed step: this rank's refined batch and its scores,
        # and the accepted rows of the whole batch (the padding past the count is undefined and left out)
        dump_outputs(args.dump_outputs, {"refined": x.cpu().numpy(), "scores": sig_local.cpu().numpy(),
                                         "accepted": acc[:n_acc].cpu().numpy(),
                                         "accepted_count": np.array([n_acc], dtype=np.float64)})
    value = world * batch * args.steps / total_s

    # ---- end-to-end through the public API: pinned host inputs, host outputs ------------------------------
    # Every step: H2D of its proposals (inside build_refiner, on the compute stream), the refinement + accept stage,
    # and D2H of the refined batch, the accepted rows and the statistics into pinned host memory.  The host consumes
    # step i while the GPU computes step i+1 (as the fill-up loop does): results are staged in one of two device
    # buffers and drained by a copy stream, the host waits for step i-1 after enqueueing step i.  All copies of all
    # timed steps complete inside the timed region (the last step is drained before the clock stops).
    NBUF = 2
    copy_stream = torch.cuda.Stream(device=dev)
    x_stage = [torch.empty_like(x) for _ in range(NBUF)]
    acc_stage = [torch.empty_like(acc) for _ in range(NBUF)]
    st_stage = [torch.empty(3, dtype=torch.float64, device=dev) for _ in range(NBUF)]
    out_host = [torch.empty((batch,) + tuple(arch["image_shape"]), dtype=torch.float32).pin_memory() for _ in range(NBUF)]
    acc_host = [torch.empty(tuple(acc.shape), dtype=torch.float32).pin_memory() for _ in range(NBUF)]
    stats_host = [torch.empty(4, dtype=torch.float64).pin_memory() for _ in range(NBUF)]
    staged = [torch.cuda.Event() for _ in range(NBUF)]
    drained = [torch.cuda.Event() for _ in range(NBUF)]
    e2e_steps = max(5, min(args.steps, 20))

    staged_in = [None]

    def e2e_enqueue(i):
        b = i % NBUF
        main = torch.cuda.current_stream()
        # H2D of this step's proposals: uploaded by Refiner.prefetch on its copy stream while the previous step was
        # computing (the first step uploads in line)
        h_in = staged_in[0] if staged_in[0] is not None else refiner.prefetch(h0_host)
        x, acc, cnt, sig_local = hot_path(h_in)
        staged_in[0] = refiner.prefetch(h0_host)                 # the NEXT step's proposals, overlapping this step
        if i >= NBUF:
            main.wait_event(drained[b])                          # staging buffer b was read out two steps ago
        x_stage[b].copy_(x)
        acc_stage[b].copy_(acc)
        st_stage[b].copy_(D.reduce_stats_async(cnt, sig_local.sum(), sig_local.max()))
        staged[b].record(main)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(staged[b])
            out_host[b].copy_(x_stage[b], non_blocking=True)     # D2H of the refined batch
            acc_host[b].copy_(acc_stage[b], non_blocking=True)   # D2H of the accepted samples (padded to the emit capacity)
            stats_host[b][:3].copy_(st_stage[b], non_blocking=True)   # D2H of the acceptance / score statistics
            drained[b].record(copy_stream)

    def e2e_collect(i):
        drained[i % NBUF].synchronize()                          # the ONE host sync per step: step i is on the host
        return stats_host[i % NBUF]

    def e2e_run(n, marks=None):
        for i in range(n):
            e2e_enqueue(i)
            if i > 0:
                e2e_collect(i - 1)
                if marks is not None:
                    marks.append(time.perf_counter())
        e2e_collect(n - 1)
        staged_in[0] = None                                      # (one upload more than steps: the last prefetch is dropped)
        if marks is not None:
            marks.append(time.perf_counter())

    e2e_run(3)                            # same call sequence as the timed loop (lazy kernel loading, allocator)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    e2e_marks = [t0]
    e2e_run(e2e_steps, e2e_marks)
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = world * batch * e2e_steps / float(e2e_t.item())
    h2d = h0_host.numel() * 4
    d2h = out_host[0].numel() * 4 + acc_host[0].numel() * 4 + 3 * 8

    line = None
    if rank == 0:
        flops_sample = S.refine_flops_per_sample(arch, ksteps)
        roof = None
        if not args.no_roofline:
            roof = build_roofline(torch, spec, arch, arch_name, batch, args.math, dev, ksteps, total_s / args.steps)
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            # N = 1 only: under torchrun the other ranks would spin in an NCCL barrier while rank 0 does host work
            sample_b = cpu_sample_rows(arch_name, ksteps)
            t = min(cpu_port_step(arch_name, gain, sample_b, ksteps, method, rate, seed=i) for i in range(2))
            cpu = {"value": sample_b / t, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                   "sample": "%d rows x K=%d (+MH), best of 2, torch-CPU FP32 oracle port" % (sample_b, ksteps)}
        _, _, bf16_sus, psrc = measured_peaks()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32" if args.math == "tf32" else "f32", "data": "synthetic",
            "config": {"workload": "%s: refine K=%d %s rate %.2g + MH(T=20), batch %d/GPU" % (arch_name, ksteps, method, rate, batch),
                       "global_batch": world * batch, "parallelism": "dp%d (sharded batch, no collective in the K loop)" % world,
                       "l2": "flushed (256 MiB write) between timed iterations; per-step working set also exceeds L2",
                       "weights": "random init seed 2019, gain %.1f" % gain,
                       "launch": "eager" if args.no_graph else "CUDA graph replay of the K-step kernel sequence",
                       "gflop_per_sample": round(flops_sample / 1e9, 3)},
            "tflops_algorithmic": round(world * batch * flops_sample / (total_s / args.steps) / 1e12, 2),
            "frac_of_tf32_peak_sustained": round(batch * flops_sample / (total_s / args.steps) / 1e12 / (0.5 * bf16_sus), 4),
            "accepted_per_step": int(n_acc),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps,
                    "pipelining": "H2D of step i+1 (Refiner.prefetch, copy stream) and D2H of step i-1 (two staging buffers, "
                                  "copy stream) overlap the compute of step i; every step's inputs come from pinned host "
                                  "memory and its outputs are in pinned host memory before the clock stops",
                    "ms_per_step_median": round(sorted(b - a for a, b in zip(e2e_marks, e2e_marks[1:]))[e2e_steps // 2] * 1e3, 3),
                    "ms_per_step_max": round(max(b - a for a, b in zip(e2e_marks, e2e_marks[1:])) * 1e3, 3)},
            "gpu_launches": int(launches * args.steps),
            "gpu_launches_per_step": int(launches),
            "clocks": clk,
        }
        if world == 1 and not args.no_extra:
            # the other BASELINE configurations on the same code path, with real step counts
            also = {}
            try:
                del flush
                torch.cuda.empty_cache()
                if args.workload != "mnist":
                    also["mnist"] = measure_extra(torch, "mnist", dev, args.math, max(args.steps, 5), max(args.warmup, 3))
                elif args.workload != "dcgan64_l1":
                    also["dcgan64_l1"] = measure_extra(torch, "dcgan64_l1", dev, args.math, max(args.steps, 5), max(args.warmup, 3))
                also["synthetic2d"] = measure_2d(torch, dev, cpu=not args.no_cpu_baseline)
                also["early_exit"] = measure_early_exit(torch, spec, arch, h0_dev, ksteps, method, rate, dev)
            except RuntimeError as exc:        # e.g. out of memory on a shared box: never lose the headline line
                also["error"] = str(exc)[:200]
            line["also"] = also
        if roof:
            line["roofline"] = roof
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


# ----------------------------------------------------------------------------------------------------------
# sweep: BASELINE configs C3 / C4 / C5 at this world size
# ----------------------------------------------------------------------------------------------------------
def sweep_points(world):
    pts = []
    pts.append(dict(config="C3", workload="dcgan32_l1", batch_total=1024 * world, k=50, scaling="weak"))
    for layer in (1, 2, 3, 4):
        pts.append(dict(config="C4", workload="dcgan64_l%d" % layer, batch_total=1024 * world, k=50, scaling="weak"))
    for wl in ("mnist", "dcgan64_l1"):
        for b in (256, 4096, 65536):
            for k in (10, 50, 200):
                pts.append(dict(config="C5", workload=wl, batch_total=b, k=k, scaling="strong"))
    return pts


def run_sweep(args):
    import numpy as np
    import torch
    from cgs import dist as D
    from cgs import nets as N
    from cgs import synthetic as S
    from sampling.collaborator import Refiner
    from sampling.idpsampler import IndependenceSampler
    dist, rank, local_rank, world, dev = setup_dist(torch)
    results = []
    specs = {}
    est_tflops = {"mnist": 200.0, "dcgan32_l1": 250.0}            # rough per-GPU rates, only to bound the run time
    for pt in sweep_points(world):
        arch_name, _, _, method, rate, gain = WORKLOADS[pt["workload"]]
        arch = N.get_arch(arch_name)
        batch = pt["batch_total"] // world
        flops = S.refine_flops_per_sample(arch, pt["k"]) * batch
        est_s = flops / (est_tflops.get(arch_name, 380.0) * 1e12)
        row = dict(pt, n_gpus=world, batch_per_gpu=batch)
        if batch < 1 or est_s > args.sweep_max_seconds:
            row["skipped"] = "estimated %.0f s per step" % est_s if batch >= 1 else "fewer rows than GPUs"
            results.append(row)
            continue
        if arch_name not in specs:
            specs.clear()                                        # one resident spec at a time
            torch.cuda.empty_cache()
            specs[arch_name] = N.NetSpec(arch, S.init_weights(arch, seed=2019, gain=gain), dev, math=args.math)
        spec = specs[arch_name]
        refiner = Refiner(pt["k"], rate, method, cuda_graph=True)
        refiner.chunk_rows = MAX_ROWS_PER_LAUNCH
        refiner.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        mh = IndependenceSampler(T=20, rng="philox", seed=2019)
        mh.set_score_curr(np.float32(0.5))
        h0 = torch.from_numpy(S.proposal_features(arch, batch, seed=1000 + rank)).to(dev)
        hot = make_hot_path(torch, D, refiner, mh, world, rank, batch)
        steps, warmup = (5, 3) if est_s < 0.5 else ((2, 1) if est_s < 8 else (1, 1))
        try:
            total_s, out = timed_steps(torch, dist, hot, h0, steps, warmup, world, None)
            t = total_s / steps
            row.update(steps=steps, warmup=warmup, ms_per_step=round(t * 1e3, 3),
                       value=round(pt["batch_total"] / t, 1), unit=UNIT,
                       tflops_algorithmic=round(world * flops / t / 1e12, 1), accepted=int(out[2].item()),
                       chunk_rows=min(batch, MAX_ROWS_PER_LAUNCH))
        except RuntimeError as exc:
            row["error"] = str(exc)[:200]
        results.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
        del refiner, mh, h0, hot
        torch.cuda.empty_cache()
    if rank == 0:
        out_dir = os.path.join(ROOT, "gpurun_out")
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, "sweep_N%d.json" % world), "w") as f:
            json.dump({"n_gpus": world, "math": args.math, "timing": "CUDA events per step, max over ranks, device-timed "
                       "(inputs resident), MH(T=20) accept + gathers inside the step", "rows": results}, f, indent=1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    wl = list(WORKLOADS[args.workload])
    if args.batch:
        wl[1] = args.batch
    if args.refine_steps:
        wl[2] = args.refine_steps
    if args.impl == "reference":
        run_reference(args, wl)
    elif args.sweep:
        run_sweep(args)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
