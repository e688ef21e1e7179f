"""Which kernels a refinement launches, in order: the route of every image-edge pass (paired mma.sync kernel, separate
mma.sync kernels, tcgen05 kernels over the space-to-depth image, general lowerings) of every shipped net.  A change of
route still passes every tolerance test; these tables catch it.  They were recorded on a B200 (TF32 mode, two
refinement steps, batch 4).
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _kernel(name):
    """'void cgs::(anonymous namespace)::edge_wide_tc_kernel<18, 2>(cgs::...)' -> 'edge_wide_tc_kernel<18,2>'"""
    depth = 0
    for i in range(len(name) - 1, -1, -1):        # cut the parameter list: the last top-level parentheses
        depth += {")": 1, "(": -1}.get(name[i], 0)
        if depth == 0 and name[i] == "(":
            name = name[:i]
            break
    name = name.replace("(anonymous namespace)::", "").replace("cgs::", "")
    return (name[5:] if name.startswith("void ") else name).replace(" ", "")


def _launched(spec, h0, flags, K=2):
    """Names of the cgs kernels one Refiner.build_refiner call launches under the CGS_DEBUG knobs `flags`."""
    from cgs import lib as L
    from cgs import nets as N
    from sampling.collaborator import Refiner
    with L.debug_flags(flags):
        r = Refiner(K, 0.1)
        r.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
        r.build_refiner(h0)                       # first launches: module loads, smem attributes
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            r.build_refiner(h0)
            torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "cgs::" in e.name),
                key=lambda e: e.time_range.start)
    return [_kernel(e.name) for e in ev]


ROUTES = {
    ('mnist', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_pair_kernel<2,1,0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_pair_kernel<2,1,1,true> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_pair_kernel<2,1,0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_pair_kernel<2,1,1,true> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_pair_kernel<2,1,0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('mnist', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('mnist', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<2,1> edge_wide_kernel<0,true> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<2,1> '
        'edge_wide_kernel<1,true> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_kernel<2,1> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<2,1> edge_wide_kernel<1,true> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<2,1> '
        'edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('mnist_l2', '0'): (
        'edge_pair_kernel<2,1,0,true> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_pair_kernel<2,1,2,false> edge_pair_kernel<2,1,0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_pair_kernel<2,1,2,false> edge_pair_kernel<2,1,0,true> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('mnist_l2', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('mnist_l2', 'NO_EDGE_PAIR'): (
        'edge_narrow_kernel<2,1> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<2,1> edge_wide_kernel<2,false> '
        'edge_narrow_kernel<2,1> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<2,1> edge_wide_kernel<2,false> '
        'edge_narrow_kernel<2,1> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<256,3,1,1,1> head_kernel '
    ).split(),
    ('dcgan32_l1', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<18> '
        'edge_wide_tc_kernel<18,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<18> '
        'edge_wide_tc_kernel<18,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan32_l1', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan32_l1', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<18> '
        'edge_wide_tc_kernel<18,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<18> '
        'edge_wide_tc_kernel<18,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<18> edge_wide_tc_kernel<18,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan48_l1', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_kernel<10,3> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_kernel<10,3> edge_wide_kernel<1,true> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<10,3> '
        'edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<10,3> '
        'edge_wide_kernel<1,true> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<10,3> edge_wide_kernel<0,true> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan48_l1', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan48_l1', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_kernel<10,3> edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_kernel<10,3> edge_wide_kernel<1,true> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<10,3> '
        'edge_wide_kernel<0,true> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_kernel<10,3> '
        'edge_wide_kernel<1,true> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_kernel<10,3> edge_wide_kernel<0,true> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan64_l1', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan64_l1', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l1', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan64_l2', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l2', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel '
    ).split(),
    ('dcgan64_l2', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l3', '0'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l3', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,2,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l3', 'NO_EDGE_PAIR'): (
        'conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,1> '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> '
        'edge_wide_tc_kernel<34,1> conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l4', '0'): (
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,2> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,2> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l4', 'EDGE_GENERAL'): (
        'conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> '
        'col2im_kernel conv_gemm_tc_kernel<64,2,1,1,1> conv_gemm_tc_kernel<64,3,1,1,1> col2im_kernel '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
    ('dcgan64_l4', 'NO_EDGE_PAIR'): (
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
        'conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,2> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> '
        'head_kernel conv_gemm_tc_kernel<64,1,1,1,1> conv_gemm_tc_kernel<64,1,1,1,1> '
        'conv_gemm_tc_kernel<64,1,1,1,1> edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,2> '
        'edge_narrow_tc_kernel<34> edge_wide_tc_kernel<34,0> conv_gemm_tc_kernel<64,0,1,1,1> '
        'conv_gemm_tc_kernel<64,0,1,1,1> conv_gemm_tc_kernel<64,0,1,1,1> head_kernel '
    ).split(),
}


@pytest.mark.parametrize("knob", ["0", "EDGE_GENERAL", "NO_EDGE_PAIR"])
@pytest.mark.parametrize("arch_name", ["mnist", "mnist_l2", "dcgan32_l1", "dcgan48_l1", "dcgan64_l1", "dcgan64_l2",
                                       "dcgan64_l3", "dcgan64_l4"])
def test_edge_routes(cgs_lib, cuda_device, arch_name, knob):
    from cgs import lib as L
    from cgs import nets as N
    from cgs import synthetic as S
    arch = N.get_arch(arch_name)
    spec = N.NetSpec(arch, S.init_weights(arch, seed=7, gain=2.5), cuda_device, math="tf32")
    h0 = torch.from_numpy(S.proposal_features(arch, 4, seed=3)).to(cuda_device)
    flags = 0 if knob == "0" else getattr(L, "DEBUG_" + knob)
    assert _launched(spec, h0, flags) == ROUTES[arch_name, knob]


def test_non_square_image_takes_the_s2d_route(cgs_lib, cuda_device):
    """A 16 x 32 image: the tcgen05 edge kernels take all four passes, so the chain runs over the space-to-depth
    layout (nothing in it needs a square image), and the refinement matches the oracle."""
    from cgs import nets as N
    from oracle import graph_refiner as gr
    from oracle import nets as onets
    from sampling.collaborator import Refiner
    arch = N.get_arch("dcgan32_l4")                 # G tail: one deconv 64 -> 3 channels, then D's four convs
    h, w = 8, 16
    arch["feature_shape"], arch["image_shape"] = [h, w, 64], [2 * h, 2 * w, 3]
    arch["gtail"] = [dict(arch["gtail"][0], hin=h, win=w)]
    for i, l in enumerate(arch["d"][:-1]):
        arch["d"][i] = dict(l, hin=2 * h >> i, win=2 * w >> i)
    arch["d"][-1] = dict(arch["d"][-1], cin=(h >> 3) * (w >> 3) * 512)
    wts = onets.scale_weights_for_signal(arch, onets.init_weights(arch, seed=9), 2.5)
    spec = N.NetSpec(arch, wts, cuda_device, math="tf32")
    h0 = torch.relu(torch.randn(3, h, w, 64, generator=torch.Generator().manual_seed(2)))
    names = _launched(spec, h0.to(cuda_device), 0)
    assert any(n.startswith("edge_narrow_tc_kernel") for n in names)
    assert any(n.startswith("edge_wide_tc_kernel") for n in names)
    o = gr.build_refiner(h0, arch, wts, 3, 0.1)
    ref = Refiner(3, 0.1)
    ref.set_env(N.discriminator_spec(spec), N.feature_to_data_spec(spec), N.loss_refine)
    out = ref.build_refiner(h0.to(cuda_device), None, "deterministic")
    e_img = float(np.linalg.norm(out.cpu().double() - o["refined"].double()) / np.linalg.norm(o["refined"].double()))
    e_logit = float((ref.optimal_logit.cpu() - o["optimal_logit"]).abs().max())
    print("non-square: img rel %.2e logit abs %.2e" % (e_img, e_logit))
    assert e_img <= 1e-2                            # DESIGN.md §2: TF32 K-step images rel-L2 <= 1e-2
    assert e_logit <= 2e-2 * max(1.0, float(o["optimal_logit"].abs().max()))
