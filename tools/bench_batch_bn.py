"""Cost of the training-mode discriminator (batch-statistic BN, `discriminator_spec(spec, is_training=True)`).

For DCGAN-64 l1 and MNIST at B = 1024, K = 50 (bench.py's weights and proposals), one call alternates three modes,
each a replayed CUDA graph of `build_refiner`, device events around every call, L2 flushed before it:
  inference_fp16  inference-mode BN folded into the weights, the default operands (FP16 where the chain takes them)
  inference_tf32  the same with CGS_DEBUG_TF32_OPERANDS (TF32 operands, what the batch mode runs on)
  batch           training-mode BN
Then a separate eager run under torch.profiler, with programmatic dependent launch off so that no kernel's time includes
waiting for its predecessor, times every BN kernel, and the bytes each must move (computed from the
shapes) give its bytes/s against the 7.7 TB/s HBM3e bound.  The pre-BN tensors are written by the GEMM just before the
statistics read them, so a BN layer smaller than the 126 MB L2 is partly read from there.

    python tools/bench_batch_bn.py [--steps 6] [--warmup 2] [--out profiles]
writes <out>/batch_bn_<workload>.json with the card's name and power limit beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "collaborative-gan-sampling_b200")]

HBM_BYTES_PER_S = 7.7e12
WORKLOADS = {"dcgan64_l1": 2.5, "mnist": 3.0}       # weight gain of bench.py's workloads
# bytes each BN kernel moves per launch, in units of the layer's [rows, C] FP32 tensor (partial sums are negligible)
KERNEL_TENSORS = {"bn_stats_kernel": 1, "bn_apply_fwd_kernel": 2, "bn_bwd_reduce_kernel": 2, "bn_bwd_apply_kernel": 3,
                  "bn_merge_kernel": 0}
FORWARD_KERNELS = ("bn_stats_kernel", "bn_apply_fwd_kernel")


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, limit = [s.strip() for s in out.strip().split(",")]
        info.update(name=name, power_limit_w=float(limit))
    except Exception as e:                                   # the number is reported without it, and says so
        info["power_limit_note"] = "nvidia-smi unavailable: %s" % e
    return info


def bn_layer_bytes(arch, B):
    """FP32 bytes of every batch-BN layer's [rows, C] tensor at batch B."""
    out = []
    for L in arch["d"]:
        if L["bn"]:
            px = 1 if L["type"] == "fc" else ((L["hin"] + 1) // 2) * ((L["win"] + 1) // 2)
            out.append(4 * B * px * L["cout"])
    return out


def make_refiner(spec, K, training, flags, h0):
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    r = Refiner(K, 0.1, "momentum", cuda_graph=True)
    r.set_env(N.discriminator_spec(spec, is_training=training), N.feature_to_data_spec(spec), N.loss_refine)
    with L.debug_flags(flags):
        r.build_refiner(h0)                                 # capture
    return r


def time_modes(spec, h0, K, steps, warmup):
    import torch
    from cgs import lib as L
    modes = {"inference_fp16": (False, 0), "inference_tf32": (False, L.DEBUG_TF32_OPERANDS), "batch": (True, 0)}
    refiners = {m: make_refiner(spec, K, tr, fl, h0) for m, (tr, fl) in modes.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=h0.device)
    ms = {m: [] for m in modes}
    for it in range(warmup + steps):
        for m, r in refiners.items():                       # alternating, so drifts hit every mode alike
            with L.debug_flags(modes[m][1]):
                flush.fill_(1)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                r.build_refiner(h0)
                e.record()
                e.synchronize()
            if it >= warmup:
                ms[m].append(s.elapsed_time(e))
    del refiners, flush
    torch.cuda.empty_cache()
    return ms


def profile_kernels(spec, h0, arch, B, K=2):
    """BN kernel times of one eager batch-mode call with K steps: K + 1 forward and K backward passes.

    Programmatic dependent launch is switched off for this run: with it, a kernel becomes resident while its
    predecessor drains and waits in griddepcontrol.wait, and the profiler counts that wait as the kernel's duration.
    The batch-mode results are bit-identical either way (tests/test_batch_bn_gpu.py)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    r = Refiner(K, 0.1, "momentum")
    r.set_env(N.discriminator_spec(spec, is_training=True), N.feature_to_data_spec(spec), N.loss_refine)
    with L.debug_flags(L.DEBUG_PDL_OFF):
        r.build_refiner(h0)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r.build_refiner(h0)
            torch.cuda.synchronize()
    layers = bn_layer_bytes(arch, B)
    out = {}
    for ev in prof.events():
        name = next((k for k in KERNEL_TENSORS if k in ev.name), None)
        if name is None or ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        d = out.setdefault(name, {"launches": 0, "us": 0.0})
        d["launches"] += 1
        d["us"] += ev.device_time
    for name, d in out.items():
        passes = K + 1 if name in FORWARD_KERNELS else K
        nbytes = KERNEL_TENSORS[name] * passes * sum(layers)
        d["us_per_launch"] = d["us"] / d["launches"]
        if nbytes:
            d["bytes"] = nbytes
            d["bytes_per_s"] = nbytes / (d["us"] * 1e-6)
            d["frac_of_hbm_bound"] = round(d["bytes_per_s"] / HBM_BYTES_PER_S, 3)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    if not torch.cuda.is_available():
        raise SystemExit("bench_batch_bn needs a CUDA device")
    L.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    os.makedirs(args.out, exist_ok=True)
    gpu = card()
    for name in args.workloads.split(","):
        arch = N.get_arch(name)
        spec = N.NetSpec(arch, S.init_weights(arch, seed=2019, gain=WORKLOADS[name]), dev, math="tf32")
        h0 = torch.from_numpy(S.proposal_features(arch, args.batch, seed=7)).to(dev)
        ms = time_modes(spec, h0, args.k, args.steps, args.warmup)
        res = {"workload": "%s: refine K=%d momentum, batch %d" % (name, args.k, args.batch), "gpu": gpu,
               "timing": "replayed CUDA graph of build_refiner, device events per call, L2 flushed before each call, "
                         "the three modes alternating; %d calls each after %d warm-up rounds" % (args.steps, args.warmup),
               "modes": {}}
        for m, v in ms.items():
            med = sorted(v)[len(v) // 2]
            res["modes"][m] = {"ms_per_call_median": round(med, 3), "ms_per_call_min": round(min(v), 3),
                               "ms_per_call_max": round(max(v), 3), "ms_per_iteration": round(med / (args.k + 1), 4),
                               "calls_ms": [round(x, 3) for x in v]}
        tf32 = res["modes"]["inference_tf32"]["ms_per_call_median"]
        res["batch_over_inference_tf32"] = round(res["modes"]["batch"]["ms_per_call_median"] / tf32, 3)
        res["batch_over_inference_default"] = round(res["modes"]["batch"]["ms_per_call_median"]
                                                    / res["modes"]["inference_fp16"]["ms_per_call_median"], 3)
        res["bn_layer_bytes"] = bn_layer_bytes(arch, args.batch)
        res["bn_kernels"] = profile_kernels(spec, h0, arch, args.batch)
        res["hbm_bound_bytes_per_s"] = HBM_BYTES_PER_S
        path = os.path.join(args.out, "batch_bn_%s.json" % name)
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: v for k, v in res.items() if k != "gpu"}), flush=True)
        del spec, h0
        torch.cuda.empty_cache()
    print(json.dumps(gpu))


if __name__ == "__main__":
    main()
