"""Time the 2-D refinement (one cgs_refine_mlp2d call per rep) and put it against the FP32-FMA bound.

    python tools/profile_2d.py [N] [--nhidden 64] [--nlayers 6] [--steps 50] [--method ladam] [--reps 20] [--cluster]

Prints the card and its power limit, the kernel form, for the cluster form the shared-memory plan and the resident
clusters (tools/probes/mlp2d_cluster_plan.cu, built into a temporary directory), ms per call, points/s and the fraction
of the FP32-FMA bound.  Work per point: 2 [(K+1) + K] nh (3 + (nlayers-2) nh) FLOP.  `--cluster` runs nh = 64 on the
cluster form (CGS_DEBUG_MLP2D_CLUSTER).  One call per rep, the real-score mean passed in, so only the refinement kernel
is timed.
"""
import argparse
import os
import subprocess
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "collaborative-gan-sampling_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from cgs import lib as L  # noqa: E402
from cgs import synthetic as S  # noqa: E402
from sampling.refiner_cpu import MlpSpec, Refiner  # noqa: E402


def smi(field):
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + field, "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def cluster_plan(nh, nlayers):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "plan")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17",
                        "-I", os.path.join(ROOT, "collaborative-gan-sampling_b200", "csrc"),
                        "-I", os.path.join(ROOT, "include"), "-o", exe,
                        os.path.join(ROOT, "tools", "probes", "mlp2d_cluster_plan.cu")], check=True)
        return subprocess.run([exe, str(nh), str(nlayers)], capture_output=True, text=True).stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("n", nargs="?", type=int, default=10000)
    ap.add_argument("--nhidden", type=int, default=64)
    ap.add_argument("--nlayers", type=int, default=6)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--method", default="ladam")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cluster", action="store_true", help="nh = 64 on the cluster form")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    n, nh, nl, K = a.n, a.nhidden, a.nlayers, a.steps
    print("card %s, power limit %s W, max SM clock %s MHz" % (
        torch.cuda.get_device_name(dev), smi("power.limit"), smi("clocks.max.sm")))
    cluster = nh != 64 or a.cluster
    print("form:", "cluster" if cluster else "split (one SM per CTA)")
    if cluster:
        print("plan:", cluster_plan(nh, nl))
    ws = S.init_mlp2d(nh, nl, seed=2019, gain=1.5)
    mlp = MlpSpec(ws, dev)
    rng = np.random.RandomState(1)
    x0 = torch.from_numpy((rng.randn(n, 2) * 4).astype(np.float32)).to(dev)
    rate = 0.1 if a.method == "ladam" else 50.0
    ref = Refiner(types.SimpleNamespace(rollout_steps=K, rollout_rate=rate, rollout_method=a.method))
    ref.set_env(mlp, None, None)
    with L.debug_flags(L.DEBUG_MLP2D_CLUSTER if a.cluster else 0):
        for _ in range(3):
            ref.manipulate_sample(x0, "deterministic", real_sigmoid_mean=0.5)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(a.reps):
            ref.manipulate_sample(x0, "deterministic", real_sigmoid_mean=0.5)
        e.record()
        e.synchronize()
    ms = s.elapsed_time(e) / a.reps
    flop = 2.0 * ((K + 1) + K) * nh * (3 + (nl - 2) * nh) * n
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    clk = smi("clocks.max.sm")
    peak = sms * 128 * 2 * float(clk) * 1e6 if clk.replace(".", "").isdigit() else float("nan")
    print("n %d nhidden %d nlayers %d K %d %s: %.3f ms per call, %.3f M points/s, %.2f TFLOP/s, %.3f of the "
          "FP32-FMA bound (%.1f TFLOP/s)" % (n, nh, nl, K, a.method, ms, n / ms / 1e3, flop / ms / 1e9,
                                             flop / ms / 1e-3 / peak, peak / 1e12))


if __name__ == "__main__":
    main()
