"""The tensor-core weight gradient (mtd_conv_wgrad_tc) against fp64 at every shape of the B = 20 train step, and every
kernel instance it dispatches to.

The host plans each call (csrc/conv_tc.cu, wg_plan): 3x3 / stride-1 / pad-1 layers with an output grid of at least
8 x 8 in plain TF32 run on the halo kernel (wgrad_halo_kernel<BN>), everything else on the tap-streaming kernel
(wgrad_tc_kernel<BN, NPASS, KP>).  The Cout tile BN and the split over pixels come from a cost model, so an instance
the model never picks at the step's shapes would otherwise ship untested: test_forced_instance runs each one through
the MTD_WG_BN / MTD_WG_KSPLIT overrides at a shape of its kernel, and test_every_instance_is_tested checks, without a
GPU, that the instance list below still matches the dispatch in the source and that each shape selects its kernel.

Errors are max |a - b| / max |b| against torch.nn.grad.conv2d_weight in fp64.  Bounds: 2e-3 for plain TF32, 5e-5 for
the 3xTF32 mode."""
import ctypes
import os
import re
import sys

import pytest
import torch

from _golden_util import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_wgrad import LAYERS  # noqa: E402

DEV = "cuda"
gpu = pytest.mark.gpu
BOUND = {1: 2e-3, 3: 5e-5}

# ---- the dispatch, restated: (kernel, BN, passes) -> a shape that reaches it, and the forced split --------------------
# halo: plain TF32 only; taps: both modes.  Each entry also forces a split (ksplit > 1: memset + atomics) or none.
INSTANCES = {
    ("halo", 32, 1): ((4, 16, 16, 64, 32, 64, 3, 1, 1), 3),
    ("halo", 64, 1): ((2, 8, 16, 32, 0, 128, 3, 1, 1), 1),
    ("halo", 128, 1): ((3, 16, 8, 96, 0, 256, 3, 1, 1), 2),
    ("taps", 32, 1): ((4, 4, 4, 64, 0, 32, 3, 1, 1), 1),
    ("taps", 64, 1): ((4, 16, 16, 64, 0, 64, 4, 2, 1), 2),
    ("taps", 128, 1): ((4, 4, 4, 64, 64, 128, 3, 1, 1), 1),
    ("taps", 32, 3): ((2, 16, 16, 32, 0, 32, 3, 1, 1), 2),
    ("taps", 64, 3): ((4, 8, 8, 64, 0, 64, 4, 2, 1), 1),
    ("taps", 128, 3): ((8, 4, 4, 128, 0, 256, 3, 1, 1), 2),
}


def source_instances():
    src = open(os.path.join(ROOT, "mtd-gan_b200", "csrc", "conv_tc.cu")).read()
    body = src[src.index("int mtd_conv_wgrad_tc(const float*"):]
    body = body[:body.index("\n}\n")]
    halo = {("halo", int(bn), 1) for bn in re.findall(r"launch_wg_halo<(\d+)>", body)}
    m = re.search(r"#define WG_DISPATCH\(BN_\)(.*)", body)
    modes = [(int(p), int(kp)) for p, kp in re.findall(r"launch_wg<BN_, (\d), (\d+)>", m.group(1))]
    taps = {("taps", int(bn), p) for bn in re.findall(r"WG_DISPATCH\((\d+)\);", body) for p, _ in modes}
    return halo | taps


def test_every_instance_is_tested():
    assert source_instances() == set(INSTANCES), "wgrad dispatch changed: update INSTANCES"
    for (kind, bn, passes), ((B, H, W, C1, C2, N, k, s, p), ks) in INSTANCES.items():
        Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
        halo_shape = k == 3 and s == 1 and p == 1 and min(Ho, Wo) >= 8
        assert N % bn == 0 and (C1 + C2) % 32 == 0
        assert (kind == "halo") == (halo_shape and passes == 1), (kind, bn, passes)


def _ref(x1, x2, dz, k, s, p):
    x = x1 if x2 is None else torch.cat([x1, x2], dim=3)
    N, C = dz.shape[3], x.shape[3]
    dw = torch.nn.grad.conv2d_weight(x.permute(0, 3, 1, 2).double(), (N, C, k, k), dz.permute(0, 3, 1, 2).double(),
                                     stride=s, padding=p)
    return dw.permute(0, 2, 3, 1).reshape(N, k * k, C)


def _run(shape, passes, seed=0):
    from mtdgan_b200 import _ext
    lib = _ext.load()
    B, H, W, C1, C2, N, k, s, p = shape
    Ho, Wo = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    g = torch.Generator(device=DEV).manual_seed(seed)
    x1 = torch.randn(B, H, W, C1, device=DEV, generator=g)
    x2 = torch.randn(B, H, W, C2, device=DEV, generator=g) if C2 else None
    dz = torch.randn(B, Ho, Wo, N, device=DEV, generator=g)
    gp = torch.full((N, k * k, C1 + C2), float("nan"), device=DEV)        # every element must be written
    plan = (ctypes.c_int * 5)()
    assert lib.mtd_conv_wgrad_tc_plan(B, H, W, C1, C2, N, k, k, s, p, passes, ctypes.addressof(plan)) == 0
    rc = lib.mtd_conv_wgrad_tc(x1.data_ptr(), None if x2 is None else x2.data_ptr(), dz.data_ptr(), gp.data_ptr(), B, H, W,
                               C1, C2, N, k, k, s, p, passes, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    torch.cuda.synchronize()
    return rel_err(gp.double(), _ref(x1, x2, dz, k, s, p)), ("halo" if plan[0] else "taps", plan[1], plan[2])


@gpu
@pytest.mark.parametrize("passes", [1, 3])
@pytest.mark.parametrize("layer", LAYERS, ids=lambda l: "x".join(map(str, l[:9])))
def test_step_shape(layer, passes):
    err, plan = _run(tuple(layer[:9]), passes)
    assert err <= BOUND[passes], (layer, passes, plan, err)


@gpu
@pytest.mark.parametrize("inst", sorted(INSTANCES), ids=lambda i: f"{i[0]}_bn{i[1]}_p{i[2]}")
def test_forced_instance(inst, monkeypatch):
    (kind, bn, passes), (shape, ks) = inst, INSTANCES[inst]
    monkeypatch.setenv("MTD_WG_BN", str(bn))
    monkeypatch.setenv("MTD_WG_KSPLIT", str(ks))
    err, plan = _run(shape, passes, seed=1)
    assert plan == (kind, bn, ks), (inst, plan)
    assert err <= BOUND[passes], (inst, plan, err)
