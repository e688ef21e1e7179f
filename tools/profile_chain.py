"""Time the refinement chain as shipped: per call, and per kernel of one refinement iteration.

bench.py's roofline times every pass through the single-layer entry point on TF32 operands; this tool times the chain
that `Refiner.build_refiner` actually runs (FP16 operands where choose_operand_type gives them, the s2d image layout,
the fused epilogues).  For each workload (bench.py's weights and proposals, B = 1024, K = 50 by default):

  * per call: a replayed CUDA graph of build_refiner, device events around every call, L2 flushed before it;
    median / min / max over --calls calls after --warmup;
  * per kernel: a separate eager call with K = 2 under torch.profiler, programmatic dependent launch off (with it a
    kernel becomes resident while its predecessor drains and the profiler counts that wait as its duration); the
    launches of the middle iteration (forward passes, head, data-gradient passes) are listed in order;
  * the bytes each pass must move, from the shapes and the operand type of every tensor: its input and output
    activations, the derivative operand of a data-gradient pass, the feature and momentum of the policy step (weights
    and per-sample scalars are left out).  Which tensors are FP16 is read from the launches themselves: the
    F16ChainParams / NarrowTc16Params forms of the kernels (conv_gemm.cu, edge_tc.cu);
  * the card's name and power limit, in the same run.

    python tools/profile_chain.py [--workloads dcgan64_l1,dcgan32_l1] [--calls 8] [--out profiles/fp16_edge_after.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "collaborative-gan-sampling_b200")]

HBM_BYTES_PER_S = 7.7e12                               # HGX B200 data sheet, one GPU
WORKLOADS = {"dcgan64_l1": 2.5, "dcgan32_l1": 2.5, "mnist": 3.0}   # weight gain of bench.py's workloads


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, limit = [s.strip() for s in out.strip().split(",")]
        info.update(name=name, power_limit_w=float(limit))
    except Exception as e:                             # the number is reported without it, and says so
        info["power_limit_note"] = "nvidia-smi unavailable: %s" % e
    return info


def short_name(name):
    """'void cgs::(anonymous namespace)::edge_wide_tc_kernel<18, 2>(cgs::...)' -> 'edge_wide_tc_kernel<18,2>'"""
    depth = 0
    for i in range(len(name) - 1, -1, -1):
        depth += {")": 1, "(": -1}.get(name[i], 0)
        if depth == 0 and name[i] == "(":
            name = name[:i]
            break
    name = name.replace("(anonymous namespace)::", "").replace("cgs::", "")
    return (name[5:] if name.startswith("void ") else name).replace(" ", "")


def chain_elems(arch):
    """Per-sample elements of act[0..n] (channel stride 4 for <= 4 channels, as the library stores them) and n_gtail."""
    layers = arch["gtail"] + arch["d"][:-1]
    cs = lambda c: 4 if c <= 4 else c

    def out_hw(L):
        if L["type"] == "fc":
            return 1, 1
        if L["type"] == "deconv":
            return 2 * L["hin"], 2 * L["win"]
        return (L["hin"] + 1) // 2, (L["win"] + 1) // 2

    L0 = layers[0]
    elems = [L0["cin"] if L0["type"] == "fc" else L0["hin"] * L0["win"] * cs(L0["cin"])]
    for L in layers:
        h, w = out_hw(L)
        elems.append(h * w * cs(L["cout"]))
    return elems, len(arch["gtail"])


def operand_types(n, n_gtail, f16, edge16):
    """fwd16[i]: act[i] (layer i's forward input) is FP16; bwd16[j]: d loss / d act[j + 1] is FP16 (refine_conv.cu).
    The image act[n_gtail] and its gradient are FP32; edge16 = False is the rule without an FP16 narrow edge form,
    under which the 64-channel side of both image-edge layers stays FP32 as well."""
    fwd = [f16 and 0 < i < n and i != n_gtail and (edge16 or i != n_gtail - 1) for i in range(n + 1)]
    bwd = [f16 and 0 <= j < n and j + 1 != n_gtail and (edge16 or j != n_gtail) for j in range(n)]
    return fwd, bwd


def pass_bytes(arch, B, f16, edge16):
    """(pass, bytes, input is FP16) per launch of one iteration, in launch order: forward 0..n-1, head,
    data-gradient n-1..0."""
    elems, ng = chain_elems(arch)
    n = len(elems) - 1
    fwd, bwd = operand_types(n, ng, f16, edge16)
    size = lambda e, h: B * e * (2 if h else 4)
    out = []
    for i in range(n):
        out.append(("forward %d" % i, size(elems[i], fwd[i]) + size(elems[i + 1], fwd[i + 1] if i + 1 < n else False),
                    fwd[i]))
    # head: the last activation in, its gradient out (the kept image / feature copies are not counted)
    out.append(("head", size(elems[n], False) + size(elems[n], bwd[n - 1]), False))
    for j in range(n - 1, -1, -1):
        b = size(elems[j + 1], bwd[j])                              # d loss / d act[j + 1]
        if j > 0:
            b += size(elems[j], bwd[j - 1]) + size(elems[j], fwd[j])   # d loss / d act[j] out, act[j] as derivative
        else:
            b += 4 * size(elems[0], False)                          # policy step: feature and momentum, in and out
        out.append(("data-gradient %d" % j, b, bwd[j]))
    return out


def make_refiner(spec, K, h0, graph):
    from cgs import nets as N
    from sampling.collaborator import Refiner
    r = Refiner(K, 0.1, "momentum", cuda_graph=graph)
    r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    r.build_refiner(h0)                                # capture / first launches
    return r


def time_calls(spec, h0, K, calls, warmup):
    import torch
    r = make_refiner(spec, K, h0, True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=h0.device)
    ms = []
    for it in range(warmup + calls):
        flush.fill_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        r.build_refiner(h0)
        e.record()
        e.synchronize()
        if it >= warmup:
            ms.append(s.elapsed_time(e))
    del r, flush
    torch.cuda.empty_cache()
    return ms


def profile_iteration(spec, h0, arch, B, K=2):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from cgs import lib as L
    with L.debug_flags(L.DEBUG_PDL_OFF):
        r = make_refiner(spec, K, h0, False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r.build_refiner(h0)
            torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "cgs::" in e.name),
                key=lambda e: e.time_range.start)
    f16 = any("F16ChainParams" in e.name for e in ev)
    edge16 = any("NarrowTc16Params" in e.name for e in ev)
    passes = pass_bytes(arch, B, f16, edge16)
    per_iter = len(passes)
    res = {"fp16_operands": f16, "fp16_narrow_edge": edge16, "launches_per_call": len(ev)}
    # one launch per pass: (K + 1) forward chains and heads, K data-gradient chains (n = (per_iter - 1) / 2 passes each)
    n = (per_iter - 1) // 2
    if len(ev) != (K + 1) * (n + 1) + K * n:
        res["note"] = "launches do not map one to one onto passes (paired edge kernels / split-K reduces): listed unlabelled"
        res["call"] = [{"kernel": short_name(e.name), "us": round(e.device_time, 2)} for e in ev]
        return res
    rows, total = [], 0.0
    for (label, nbytes, in16), e in zip(passes, ev[per_iter:2 * per_iter]):
        us = e.device_time
        total += us
        row = {"pass": label, "kernel": short_name(e.name), "input": "fp16" if in16 else "fp32",
               "us": round(us, 2), "bytes": nbytes}
        if nbytes and us > 0:
            row["bytes_per_s"] = round(nbytes / (us * 1e-6), -8)
            row["frac_of_hbm_bound"] = round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 3)
        rows.append(row)
    res["iteration"] = rows
    res["iteration_us_sum"] = round(total, 1)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--calls", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--workloads", default="dcgan64_l1")
    ap.add_argument("--out", default=None, help="JSON file for the results (default: stdout only)")
    args = ap.parse_args()
    import torch
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    if not torch.cuda.is_available():
        raise SystemExit("profile_chain needs a CUDA device")
    L.load()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": card(), "hbm_bound_bytes_per_s": HBM_BYTES_PER_S,
           "timing": "per call: replayed CUDA graph of build_refiner, device events, L2 flushed before each call, "
                     "%d calls after %d warm-up calls; per kernel: eager K = 2 call under torch.profiler with "
                     "programmatic dependent launch off, its second iteration" % (args.calls, args.warmup),
           "workloads": {}}
    for name in args.workloads.split(","):
        arch = N.get_arch(name)
        spec = N.NetSpec(arch, S.init_weights(arch, seed=2019, gain=WORKLOADS[name]), dev, math="tf32")
        h0 = torch.from_numpy(S.proposal_features(arch, args.batch, seed=7)).to(dev)
        ms = time_calls(spec, h0, args.k, args.calls, args.warmup)
        med = sorted(ms)[len(ms) // 2]
        w = {"workload": "%s: refine K=%d momentum, batch %d" % (name, args.k, args.batch),
             "ms_per_call_median": round(med, 3), "ms_per_call_min": round(min(ms), 3),
             "ms_per_call_max": round(max(ms), 3), "ms_per_iteration": round(med / (args.k + 1), 4),
             "calls_ms": [round(x, 3) for x in ms]}
        w.update(profile_iteration(spec, h0, arch, args.batch))
        res["workloads"][name] = w
        print(json.dumps(w), flush=True)
        del spec, h0
        torch.cuda.empty_cache()
    print(json.dumps(res["gpu"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
