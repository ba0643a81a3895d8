"""GPU parity tests of the individual kernels, called through the C-ABI (via the ctypes host mirror),
against torch-CPU fp64 evaluations of the same operator on the same seeded inputs.
Tolerance: fp32 SIMT kernels <= 1e-5 (norm-wise relative error, max|a-b| / max|b|)."""
import math

import pytest
import torch
import torch.nn.functional as F

from _golden_util import load, rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
TOL = 1e-5


def nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def nchw(t):
    return t.permute(0, 3, 1, 2).contiguous()


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float64) * scale


CONV_CASES = [
    # B, H, W, C1, C2, N, k, s, p, transposed, pre, post, add
    (2, 16, 16, 32, 0, 32, 3, 1, 1, 0, 1, 0, False),
    (2, 16, 16, 1, 0, 32, 3, 1, 1, 0, 1, 0, False),      # Cin = 1 (generator encoder[0], conv11)
    (2, 16, 16, 32, 0, 1, 3, 1, 1, 1, 0, 1, True),       # ConvTranspose, Cout = 1, skip add + post relu
    (2, 16, 16, 32, 0, 32, 3, 1, 1, 1, 0, 1, True),      # generator decoder layer
    (2, 8, 8, 64, 64, 128, 3, 1, 1, 0, 2, 0, False),     # two sources (torch.cat skip), leaky
    (2, 16, 16, 64, 0, 64, 4, 2, 1, 0, 0, 0, False),     # down* conv: 4x4 stride 2, no activation
    (3, 1, 1, 512, 0, 512, 1, 1, 0, 0, 2, 0, False),     # bottleneck 1x1 / Linear
    (3, 2, 2, 512, 0, 512, 3, 1, 1, 0, 2, 0, False),     # skinny-M split-K
    (2, 2, 2, 512, 512, 256, 3, 1, 1, 0, 2, 0, False),   # skinny-M split-K, two sources
    (2, 4, 4, 12, 0, 20, 3, 1, 1, 0, 2, 0, False),       # channels not multiples of 4 (scalar path)
    (5, 2, 2, 64, 0, 64, 4, 2, 1, 0, 0, 0, False),       # down6-like: 2x2 -> 1x1
    (2, 64, 64, 128, 0, 1, 3, 1, 1, 0, 2, 0, False),     # s_dconv61: Cout = 1
    (2, 64, 64, 1, 0, 1, 3, 1, 1, 0, 2, 0, False),       # s_dconv62 / 1 -> 1
    (3, 64, 64, 64, 64, 1, 3, 1, 1, 0, 2, 0, False),     # s_dconv61 on cat[up, skip]: halo-tile N = 1 kernel, two sources
    (1, 64, 64, 32, 0, 1, 3, 1, 1, 1, 0, 1, True),       # generator decoder[0] (ConvTranspose 32 -> 1, skip add): N = 1 tile kernel
    (2, 64, 64, 1, 0, 64, 3, 1, 1, 0, 2, 0, False),      # conv11 1 -> 64: vectorised Cin = 1 kernel; its dgrad is the N = 1 tile kernel
    (4, 128, 128, 1, 0, 64, 3, 1, 1, 0, 2, 0, False),    # large enough for the 16-channels-per-thread Cin = 1 kernel
    (8, 128, 128, 1, 0, 32, 3, 1, 1, 0, 1, 0, False),    # the same kernel, generator conv_first shape
]


@pytest.fixture()
def exact_kernels():
    from mtdgan_b200 import ops
    ops.set_conv_mode("simt")
    yield
    ops.set_conv_mode("auto", 3)


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv_forward_backward(case, exact_kernels):
    """Exact-fp32 CUDA-core kernels (generic implicit GEMM + the thin-layer streaming kernels)."""
    from mtdgan_b200 import ops
    B, H, W, C1, C2, N, k, s, p, tr, pre, post, add = case
    C = C1 + C2
    x = _rand(B, C, H, W, seed=1)
    w = _rand(*((C, N, k, k) if tr else (N, C, k, k)), seed=2, scale=1.0 / math.sqrt(C * k * k))
    b = _rand(N, seed=3, scale=0.1)
    Ho = (H + 2 * p - k) // s + 1
    skip = _rand(B, N, Ho, Ho, seed=4) if add else None
    gout = _rand(B, N, Ho, Ho, seed=5)
    # ---- torch fp64 reference
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    sr = skip.clone().requires_grad_(True) if add else None
    act = {0: lambda t: t, 1: F.relu, 2: lambda t: F.leaky_relu(t, 0.2)}
    z = F.conv_transpose2d(xr, wr, br, padding=p) if tr else F.conv2d(xr, wr, br, stride=s, padding=p)
    yr = act[pre](z)
    if add:
        yr = yr + sr
    yr = act[post](yr)
    yr.backward(gout)
    # ---- CUDA
    xc = nhwc(x.float()).to(DEV)
    x1 = xc[..., :C1].contiguous().requires_grad_(True)
    x2 = xc[..., C1:].contiguous().requires_grad_(True) if C2 else None
    wc, bc = w.float().to(DEV).requires_grad_(True), b.float().to(DEV).requires_grad_(True)
    sc = nhwc(skip.float()).to(DEV).requires_grad_(True) if add else None
    cfg = ops.ConvCfg(cin=C, cout=N, kh=k, kw=k, stride=s, pad=p, transposed=tr, pre_act=pre, post_act=post)
    y = ops.conv(x1, wc, bc, cfg, x2=x2, add1=sc)
    y.backward(nhwc(gout.float()).to(DEV))
    torch.cuda.synchronize()
    assert rel_err(nchw(y), yr) <= TOL
    dx = nchw(x1.grad) if not C2 else torch.cat([nchw(x1.grad), nchw(x2.grad)], 1)
    assert rel_err(dx, xr.grad) <= TOL
    assert rel_err(wc.grad, wr.grad) <= TOL
    assert rel_err(bc.grad, br.grad) <= TOL
    if add:
        assert rel_err(nchw(sc.grad), sr.grad) <= TOL


TC_CASES = [
    # B, H, W, C1, C2, N, k, p, transposed, pre, post, add     (all stride 1, >= 2048 output pixels)
    (2, 64, 64, 32, 0, 32, 3, 1, 0, 1, 0, False),        # generator encoder / img_conv
    (2, 64, 64, 32, 0, 32, 3, 1, 1, 0, 1, True),         # generator decoder (ConvTranspose + skip + relu)
    (2, 32, 32, 64, 64, 128, 3, 1, 0, 2, 0, False),      # decoder conv on cat[up, skip]
    (4, 32, 32, 128, 0, 64, 1, 0, 0, 2, 0, False),       # 1x1
    (8, 16, 16, 256, 0, 256, 3, 1, 0, 2, 0, False),      # TW=16, TH=8
    (33, 8, 8, 256, 0, 512, 3, 1, 0, 2, 0, False),       # TW=8, TH=8, TB=2 with a ragged last batch tile
    (1, 32, 128, 32, 0, 32, 3, 1, 0, 1, 0, False),       # TW=128, TH=1
    (1, 8, 512, 32, 0, 64, 3, 1, 0, 1, 0, False),        # 512-wide rows (inference geometry)
    (20, 4, 4, 512, 0, 512, 3, 1, 0, 2, 0, False),       # skinny M = 320: split-K weight streaming
    (20, 2, 2, 512, 512, 512, 3, 1, 0, 2, 0, False),     # M = 80, two sources, split-K
    (20, 1, 1, 512, 0, 512, 1, 0, 0, 2, 0, False),       # bottleneck 1x1 at 1x1 spatial (TB = 128)
    (3, 4, 4, 512, 0, 2048, 1, 0, 0, 0, 0, False),       # UpsampleBlock 1x1 conv C -> 4C
    (5, 16, 8, 32, 0, 32, 3, 1, 0, 1, 0, False),         # halo-tile kernel: one 16 x 8 tile per image (all four borders padded)
    (1, 512, 512, 32, 0, 32, 3, 1, 1, 0, 1, True),       # halo-tile kernel at the inference geometry (2048 tiles, 14 per CTA)
    (3, 64, 32, 32, 0, 32, 3, 1, 0, 1, 0, False),        # halo-tile kernel, 4 x 4 tiles per image, ragged over 148 CTAs
    (20, 32, 32, 128, 0, 128, 3, 1, 0, 2, 0, False),     # streamed-weight halo kernel: 160 tiles = one wave + a stream-K wave
    (20, 16, 16, 256, 0, 256, 3, 1, 0, 2, 0, False),     # streamed-weight halo kernel: 80 tiles, all stream-K pieces
    (4, 64, 64, 64, 0, 64, 3, 1, 1, 0, 1, True),         # streamed-weight halo kernel, BN = 64, ConvTranspose + skip + relu
    (2, 16, 16, 64, 0, 32, 3, 1, 0, 1, 0, False),        # streamed-weight halo kernel, BN = 32
    (3, 16, 8, 96, 32, 64, 3, 1, 0, 2, 0, False),        # streamed-weight halo kernel, unequal two sources, one tile per image
]


@pytest.fixture(params=[1, 2], ids=["v1_smemA", "v2_tmemA"])
def tc_version(request):
    """Both generations of the forward/dgrad tensor-core kernel: v1 keeps the rounded A tile in shared memory (whole-tile
    waves + stream-K wave), v2 writes it to TMEM (tcgen05.st) and shares every weight stage among several pixel tiles."""
    from mtdgan_b200 import ops
    prev = ops.set_tc_version(request.param)
    yield request.param
    ops.set_tc_version(prev)


@pytest.mark.parametrize("passes,tol", [(1, 2e-3), (3, 5e-5)], ids=["tf32", "tf32x3"])
@pytest.mark.parametrize("B,H,C", [(2, 64, 64), (20, 8, 512), (20, 2, 512), (3, 16, 256)])
def test_conv_tcgen05_stride2(B, H, C, passes, tol, tc_version):
    """down* layers (4x4, stride 2, pad 1) on the tcgen05 kernels: forward and wgrad through TMA element strides,
    data gradient as four output-parity classes."""
    from mtdgan_b200 import ops
    x = _rand(B, C, H, H, seed=1)
    w = _rand(C, C, 4, 4, seed=2, scale=1.0 / math.sqrt(C * 16))
    b = _rand(C, seed=3, scale=0.1)
    gout = _rand(B, C, H // 2, H // 2, seed=5)
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yr = F.conv2d(xr, wr, br, stride=2, padding=1)
    yr.backward(gout)
    xc = nhwc(x.float()).to(DEV).requires_grad_(True)
    wc, bc = w.float().to(DEV).requires_grad_(True), b.float().to(DEV).requires_grad_(True)
    cfg = ops.ConvCfg(cin=C, cout=C, kh=4, kw=4, stride=2, pad=1)
    ops.set_conv_mode("auto", passes)
    ops.set_wgrad_passes(passes)
    try:
        n0 = ops.tc_launches
        y = ops.conv(xc, wc, bc, cfg)
        y.backward(nhwc(gout.float()).to(DEV))
        torch.cuda.synchronize()
        assert ops.tc_launches - n0 == 3, "tcgen05 fwd / dgrad / wgrad were not all selected"
    finally:
        ops.set_conv_mode("auto", 3)
        ops.set_wgrad_passes(1)
    assert rel_err(nchw(y), yr) <= tol
    assert rel_err(nchw(xc.grad), xr.grad) <= tol
    assert rel_err(wc.grad, wr.grad) <= tol
    assert rel_err(bc.grad, br.grad) <= 2e-5


@pytest.mark.parametrize("passes,tol", [(1, 2e-3), (3, 5e-5)], ids=["tf32", "tf32x3"])
@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: "x".join(map(str, c)))
def test_conv_tcgen05_forward_backward(case, passes, tol, tc_version):
    """tcgen05/TMEM kernel (forward + dgrad) vs fp64 torch: plain TF32 <= 2e-3, error-compensated 3xTF32 <= 2e-5;
    and it must really be the kernel that ran.  The backward reference uses the activation mask of the CUDA
    forward (a ReLU sign flip at |z| ~ 1e-3 is not a kernel error; the mask kernels are tested on their own)."""
    from mtdgan_b200 import ops
    B, H, W, C1, C2, N, k, p, tr, pre, post, add = case
    C = C1 + C2
    x = _rand(B, C, H, W, seed=1)
    w = _rand(*((C, N, k, k) if tr else (N, C, k, k)), seed=2, scale=1.0 / math.sqrt(C * k * k))
    b = _rand(N, seed=3, scale=0.1)
    skip = _rand(B, N, H, W, seed=4) if add else None
    gout = _rand(B, N, H, W, seed=5)
    act = {0: lambda t: t, 1: F.relu, 2: lambda t: F.leaky_relu(t, 0.2)}
    dact = {0: lambda y: torch.ones_like(y), 1: lambda y: (y > 0).double(), 2: lambda y: torch.where(y > 0, 1.0, 0.2).double()}
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    z = F.conv_transpose2d(xr, wr, br, padding=p) if tr else F.conv2d(xr, wr, br, padding=p)
    yr = act[pre](z)
    if add:
        yr = yr + skip
    yr = act[post](yr)
    xc = nhwc(x.float()).to(DEV)
    x1 = xc[..., :C1].contiguous().requires_grad_(True)
    x2 = xc[..., C1:].contiguous().requires_grad_(True) if C2 else None
    wc, bc = w.float().to(DEV).requires_grad_(True), b.float().to(DEV).requires_grad_(True)
    sc = nhwc(skip.float()).to(DEV).requires_grad_(True) if add else None
    cfg = ops.ConvCfg(cin=C, cout=N, kh=k, kw=k, stride=1, pad=p, transposed=tr, pre_act=pre, post_act=post)
    ops.set_conv_mode("auto", passes)
    ops.set_wgrad_passes(passes)
    try:
        n0 = ops.tc_launches
        y = ops.conv(x1, wc, bc, cfg, x2=x2, add1=sc)
        y.backward(nhwc(gout.float()).to(DEV))
        torch.cuda.synchronize()
        # a torch.cat layer's two data gradients come from one launch on the v1 kernel, from two on v2
        assert ops.tc_launches - n0 == (4 if (C2 and tc_version == 2) else 3), "tcgen05 kernels (fwd, dgrad, wgrad) were not all selected"
    finally:
        ops.set_conv_mode("auto", 3)
        ops.set_wgrad_passes(1)
    assert rel_err(nchw(y), yr) <= tol
    # backward reference through the CUDA forward's own activation pattern
    yc = nchw(y).detach().double().cpu()
    g1 = gout * dact[post](yc)
    pre_out = yc if not add else act[pre](z.detach())           # pre_act is NONE whenever a skip is added here
    dz = g1 * dact[pre](pre_out)
    z.backward(dz)
    dx = nchw(x1.grad) if not C2 else torch.cat([nchw(x1.grad), nchw(x2.grad)], 1)
    assert rel_err(dx, xr.grad) <= tol
    assert rel_err(wc.grad, wr.grad) <= tol                     # tcgen05 wgrad (MN-major operands, split-K over pixels)
    assert rel_err(bc.grad, br.grad) <= 2e-5
    if add:
        assert rel_err(nchw(sc.grad), g1) <= 1e-6


def test_conv_weight_grad_filter_and_frozen_weights():
    from mtdgan_b200 import ops
    x = nhwc(_rand(2, 8, 8, 8, seed=1).float()).to(DEV).requires_grad_(True)
    w = _rand(8, 8, 3, 3, seed=2).float().to(DEV).requires_grad_(True)
    b = torch.zeros(8, device=DEV, requires_grad=True)
    cfg = ops.ConvCfg(cin=8, cout=8)
    y = ops.conv(x, w, b, cfg)
    with ops.wgrad_only_for([b]):
        gx, gw = torch.autograd.grad(y.sum(), [x, w], allow_unused=True, retain_graph=True)
    assert gx is not None and gw is None
    gx2, gw2 = torch.autograd.grad(y.sum(), [x, w])
    assert gw2 is not None and torch.equal(gx, gx2)
    import dataclasses
    y2 = ops.conv(x, w, b, dataclasses.replace(cfg, freeze=True))
    gx3, gw3, gb3 = torch.autograd.grad(y2.sum(), [x, w, b], allow_unused=True)
    assert torch.equal(gx3, gx2) and gw3 is None and gb3 is None


def test_spectral_norm_conv_matches_torch():
    """D-style SN conv: power iteration, 1/sigma epilogue and the analytic SN backward (SURVEY A4/A5)."""
    import torch.nn as nn
    from mtdgan_b200 import networks as NW
    torch.manual_seed(3)
    ref = nn.utils.spectral_norm(nn.Conv2d(16, 24, 3, 1, 1)).double()
    x = _rand(2, 16, 8, 8, seed=4)
    sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
    ref.train()
    xr = x.clone().requires_grad_(True)
    yr = F.leaky_relu(ref(xr), 0.2)
    gout = _rand(*yr.shape, seed=5)
    yr.backward(gout)
    # drive the same kernels through a minimal stand-in: one SN layer registered like the discriminator's
    holder = nn.Module()
    holder.conv = nn.utils.spectral_norm(nn.Conv2d(16, 24, 3, 1, 1))
    holder.conv.load_state_dict({k: v.float() for k, v in sd0.items()})
    holder.to(DEV)
    st = NW._SNState([holder.conv], torch.device(DEV))
    from mtdgan_b200._ext import call, fptr, ptr, stream
    from mtdgan_b200 import ops
    u_snap = torch.empty(st.u_total, device=DEV)
    v_snap = torch.empty(st.v_total, device=DEV)
    inv = torch.empty(1, device=DEV)
    call("mtd_sn_power_iter", ptr(st.tab), 1, ptr(st.wtu), st.n_wtu, ptr(st.wv), st.n_wv, fptr(st.t_ws), st.t_elems,
         fptr(st.s_ws), fptr(u_snap), fptr(v_snap), fptr(inv), 1, 1e-12, stream())
    xc = nhwc(x.float()).to(DEV).requires_grad_(True)
    cfg = ops.ConvCfg(cin=16, cout=24, pre_act=ops.ACT_LEAKY)
    y = ops.conv(xc, holder.conv.weight_orig, holder.conv.bias, cfg, inv_sigma=inv, u=u_snap, v=v_snap)
    y.backward(nhwc(gout.float()).to(DEV))
    torch.cuda.synchronize()
    assert rel_err(holder.conv.weight_u, ref.weight_u) <= TOL and rel_err(holder.conv.weight_v, ref.weight_v) <= TOL
    assert rel_err(nchw(y), yr) <= TOL
    assert rel_err(nchw(xc.grad), xr.grad) <= TOL
    assert rel_err(holder.conv.weight_orig.grad, ref.weight_orig.grad) <= 2e-5
    assert rel_err(holder.conv.bias.grad, ref.bias.grad) <= TOL


@pytest.mark.parametrize("B,H,W,C", [(2, 1, 1, 8), (2, 2, 2, 16), (1, 8, 8, 5), (2, 32, 32, 64)])
def test_upsample_bilinear(B, H, W, C):
    from mtdgan_b200 import ops
    x = _rand(B, C, H, W, seed=7)
    xr = x.clone().requires_grad_(True)
    yr = F.interpolate(xr, scale_factor=2, mode="bilinear", align_corners=False)
    g = _rand(*yr.shape, seed=8)
    yr.backward(g)
    xc = nhwc(x.float()).to(DEV).requires_grad_(True)
    y = ops.Upsample2xFn.apply(xc)
    y.backward(nhwc(g.float()).to(DEV))
    assert rel_err(nchw(y), yr) <= 1e-6 and rel_err(nchw(xc.grad), xr.grad) <= 1e-6


def test_pixel_shuffle_layout_clip_mul():
    from mtdgan_b200 import ops
    x = _rand(2, 32, 4, 4, seed=9)
    xr = x.clone().requires_grad_(True)
    yr = F.pixel_shuffle(xr, 2)
    g = _rand(*yr.shape, seed=10)
    yr.backward(g)
    xc = nhwc(x.float()).to(DEV).requires_grad_(True)
    y = ops.PixelShuffle2Fn.apply(xc)
    y.backward(nhwc(g.float()).to(DEV))
    assert torch.equal(nchw(y).cpu(), yr.float()) and torch.equal(nchw(xc.grad).cpu(), xr.grad.float())
    # layout transposes are exact permutations
    t = torch.randn(3, 5, 7, 9, device=DEV)
    assert torch.equal(ops.to_nhwc(t), t.permute(0, 2, 3, 1).contiguous())
    assert torch.equal(ops.to_nchw(ops.to_nhwc(t)), t)
    # clip(0,1): closed-interval gradient (SURVEY A10)
    v = torch.tensor([-0.5, 0.0, 0.25, 1.0, 1.5, -0.0], device=DEV).requires_grad_(True)
    c = ops.Clip01Fn.apply(v)
    c.backward(torch.ones_like(v))
    assert c.tolist() == [0.0, 0.0, 0.25, 1.0, 1.0, 0.0] and v.grad.tolist() == [0, 1, 1, 1, 0, 1]


@pytest.mark.parametrize("mode", ["simt", "auto"])
def test_fft_block_vs_golden_and_oracle(mode):
    """FFT_ConvBlock forward + all gradients against the golden vectors from the live reference.  "simt": exact fp32
    everywhere (1e-4 on everything); "auto" (default): the img_conv runs on tcgen05 (3xTF32 forward / dgrad: still
    1e-4; plain-TF32 weight gradient: the north_star's tensor-core bound 2e-3)."""
    from arch.Ours.networks import FFT_ConvBlock
    from mtdgan_b200 import ops
    ops.set_conv_mode(mode, 3 if mode == "auto" else None)
    try:
        torch.manual_seed(5)
        blk = FFT_ConvBlock(32).to(DEV)
        g = torch.Generator().manual_seed(6)
        x = (0.5 * torch.randn(1, 32, 64, 64, generator=g)).to(DEV).requires_grad_(True)
        wgt = torch.randn(1, 32, 64, 64, generator=g).to(DEV)
        out = blk(x)
        (out * wgt).sum().backward()
    finally:
        ops.set_conv_mode("auto", 3)
    fix = load("fftblock_64.pt")
    assert rel_err(out, fix["out"]) <= 1e-4          # north_star: fp32 rel. error <= 1e-4 on FFT/conv outputs
    assert rel_err(x.grad, load("fftblock_64_dx.pt")["dx"]) <= 1e-4
    for k, p in blk.named_parameters():
        tol = 2e-3 if (mode == "auto" and k == "img_conv.weight") else 1e-4
        assert rel_err(p.grad, fix["grads"][k]) <= tol, k


# (B, H, W) of the four-step row transforms: every length 64 ... 512; at W = 64 a CTA takes two rows, and an odd B*H
# (63, 21) leaves the last CTA half filled
FFT_ROW_CASES = [(1, 64, 64), (1, 128, 64), (1, 64, 128), (1, 64, 256), (1, 512, 512), (1, 63, 64), (3, 7, 64), (2, 33, 512)]


@pytest.mark.parametrize("B,H,W", FFT_ROW_CASES)
def test_fft_rows_roundtrip_and_rfft(B, H, W):
    """Row transforms: irfft_W(rfft_W(x)) == x, and the half spectrum equals torch.fft.rfft along W in fp64."""
    from mtdgan_b200._ext import call, fptr, stream, load as libload
    C = 32
    x = torch.randn(B, H, W, C, generator=torch.Generator().manual_seed(B * 100000 + H * 1000 + W)).to(DEV)
    spec = torch.empty(libload().mtd_fft_spec_elems(B, H, W, C), device=DEV)
    call("mtd_fft_rows_fwd", fptr(x), fptr(spec), B, H, W, C, stream())
    back = torch.empty_like(x)
    call("mtd_fft_rows_inv", fptr(spec), None, None, fptr(back), B, H, W, C, stream())
    want = torch.fft.rfft(x.double().cpu(), dim=2, norm="ortho")            # (B,H,Wh,C)
    got = torch.view_as_complex(spec.view(B, W // 2 + 1, H, C, 2)).permute(0, 2, 1, 3).cpu()
    fwd = float((got - want).abs().max() / want.abs().max())
    inv = rel_err(back, x)
    print("rows B=%d H=%d W=%d: rfft err %.2e, roundtrip err %.2e" % (B, H, W, fwd, inv))
    assert inv <= 2e-6 and fwd <= 2e-6


def test_losses_vs_golden_and_mask_bit_exact():
    import losses as LS
    from oracle import mtdgan_oracle as O
    fix = load("losses.pt")
    xs, ys = O.synthetic_pair(4, 64, seed=32)
    xs, ys = xs.to(DEV), ys.to(DEV)
    fns = {"ls_gan1": lambda p: LS.ls_gan(p, 1.0), "nds0": lambda p: LS.NDS_Loss(p, 0.0, xs - ys),
           "charb": lambda p: LS.CharbonnierLoss()(p, ys), "edge": lambda p: LS.EdgeLoss()(p, ys)}
    for name, fn in fns.items():
        p = fix["pred"].to(DEV).requires_grad_(True)
        v = fn(p)
        v.backward()
        assert abs(float(v) - float(fix[name]["value"])) <= 1e-5 * abs(float(fix[name]["value"])), name
        # edge/charbonnier gradients are d/sqrt(d^2+eps^2) with eps = 1e-3: fp32 evaluation-order noise in d
        # (~1e-7) is amplified by 1/eps, so the north_star's 1e-4 is the meaningful bound here
        assert rel_err(p.grad, fix[name]["grad"]) <= (1e-4 if name in ("edge", "charb") else 1e-5), name
    m = LS.nds_mask(fix["spec"].to(DEV), fix["ysp"].to(DEV))
    assert torch.equal(m.cpu(), fix["mask_special"])                       # bit-exact incl. -0.0 / denormal / NaN
    big_x, big_y = O.synthetic_pair(20, 64, seed=1234)
    assert torch.equal(LS.nds_mask(big_x.to(DEV), big_y.to(DEV)).cpu(), O.nds_mask(big_x - big_y))


def test_pcgrad_demo_known_answer_on_gpu():
    """The reference's own self-check (module/pcgrad.py:165-195) through the CUDA PCGrad."""
    from module.pcgrad import run_demo
    from test_oracle import _DEMO_PRINTED
    got = run_demo(DEV)
    gold = load("pcgrad_demo.pt")["grads"]
    for net_got, net_gold, net_print in zip(got, gold, _DEMO_PRINTED):
        for a, b, c in zip(net_got, net_gold, net_print):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)
            assert torch.allclose(a, torch.tensor(c), atol=6e-5)


def test_pcgrad_full_size_properties():
    """At the discriminator's real size (28.6 M shared floats, 40 segments): Gram matches fp64 torch, the
    merged gradient equals sum_k coef_k g_k, and with no conflicts PCGrad degenerates to the plain sum."""
    import random
    from mtdgan_b200.weight_methods import pcgrad_merge, draw_visit_orders
    from oracle import mtdgan_oracle as O
    sizes = [64, 576, 64, 36864, 65536, 73728, 147456, 262144, 2359296, 4194304, 512, 9437184 // 4]
    g = torch.Generator(device=DEV).manual_seed(0)
    base = [torch.randn(n, device=DEV, generator=g) for n in sizes]
    t0 = [b.clone() for b in base]
    t1 = [-0.5 * b + 0.3 * torch.randn(b.shape, device=DEV, generator=g) for b in base]     # conflicts with t0
    t2 = [1e-5 * torch.randn(b.shape, device=DEV, generator=g) for b in base]                # tiny, like task 2
    random.seed(5)
    orders = draw_visit_orders(3)
    merged, dbg = pcgrad_merge([t0, t1, t2], orders, mean=False, return_debug=True)
    flat = [torch.cat(t).double() for t in (t0, t1, t2)]
    gram = torch.stack([torch.stack([a @ b for b in flat]) for a in flat]).cpu()
    assert torch.allclose(dbg["gram"].cpu(), gram, rtol=1e-9)
    C = O.pcgrad_coefficients(gram.numpy(), orders)
    assert torch.allclose(dbg["C"].double().cpu(), torch.tensor(C), rtol=1e-5, atol=1e-7)
    want = sum(float(C.sum(0)[k]) * flat[k] for k in range(3))
    got = torch.cat([m.flatten() for m in merged]).double()
    assert float((got - want).norm() / want.norm()) <= 1e-6
    merged2 = pcgrad_merge([t0, [2 * b for b in t0]], [[0, 1], [1, 0]], mean=False)
    assert rel_err(torch.cat(merged2), 3 * torch.cat(t0)) <= 1e-6


def test_adamw_step_matches_torch():
    from mtdgan_b200.optim import FusedAdamW
    torch.manual_seed(0)
    ps = [torch.randn(n, device=DEV) for n in (5, 1000, 40000)]
    a = [p.clone().requires_grad_(True) for p in ps]
    b = [p.clone().requires_grad_(True) for p in ps]
    oa = torch.optim.AdamW(a, lr=1e-3, weight_decay=5e-4)
    ob = FusedAdamW(b, lr=1e-3, weight_decay=5e-4)
    for it in range(3):
        for i, (pa, pb) in enumerate(zip(a, b)):
            g = torch.randn(pa.shape, device=DEV)
            pa.grad = None if (i == 0 and it == 1) else g.clone()
            pb.grad = None if (i == 0 and it == 1) else g.clone()
        oa.step()
        ob.step()
    for pa, pb in zip(a, b):
        assert rel_err(pb, pa) <= 1e-6


@pytest.mark.parametrize("M,N,groups,act", [(16, 512, 1, 2), (40, 512, 2, 2), (2 * 3 * 64 * 64, 64, 2, 2), (8, 2048, 2, 0), (6 * 17, 24, 2, 2)])
def test_act_bwd_sn_matches_reference(M, N, groups, act):
    """mtd_act_bwd_sn: dz, bias gradient and the per-call spectral-norm coefficients sum dz.(y_pre - b)."""
    from mtdgan_b200._ext import call, fptr, stream
    g = torch.Generator().manual_seed(M + N)
    ypre = torch.randn(M, N, generator=g, dtype=torch.float64)
    bias = torch.randn(N, generator=g, dtype=torch.float64) * 0.1
    dy = torch.randn(M, N, generator=g, dtype=torch.float64)
    y = torch.where(ypre > 0, ypre, 0.2 * ypre) if act == 2 else ypre
    dz_ref = dy * torch.where(y > 0, 1.0, 0.2) if act == 2 else dy
    zw_ref = (dz_ref * (ypre - bias)).reshape(groups, -1).sum(1)
    dyc, yc, bc = dy.float().to(DEV), y.float().to(DEV), bias.float().to(DEV)
    dz = torch.empty_like(dyc)
    db = torch.zeros(N, device=DEV)
    zw = torch.zeros(groups, dtype=torch.float64, device=DEV)
    call("mtd_act_bwd_sn", fptr(dyc), fptr(yc), fptr(dz), fptr(db), fptr(bc), zw.data_ptr(), None, groups, M, N, act, 0.2, stream())
    torch.cuda.synchronize()
    assert rel_err(dz, dz_ref) <= 1e-6
    # pre-scaled dz (1/sigma per batched call); bias gradient and coefficients stay unscaled
    sc = torch.tensor([0.5 + 0.25 * g_ for g_ in range(groups)], device=DEV)
    dz2, db2 = torch.empty_like(dyc), torch.zeros(N, device=DEV)
    zw2 = torch.zeros(groups, dtype=torch.float64, device=DEV)
    call("mtd_act_bwd_sn", fptr(dyc), fptr(yc), fptr(dz2), fptr(db2), fptr(bc), zw2.data_ptr(), fptr(sc), groups, M, N, act, 0.2,
         stream())
    torch.cuda.synchronize()
    want = (dz_ref.reshape(groups, -1) * sc.double().cpu().reshape(groups, 1)).reshape(M, N)
    assert rel_err(dz2, want) <= 1e-6 and rel_err(db2, dz_ref.sum(0)) <= 1e-5
    assert float((zw2.cpu() - zw_ref).abs().max()) <= 2e-6 * float((dz_ref * (ypre - bias)).abs().reshape(groups, -1).sum(1).max())
    assert rel_err(db, dz_ref.sum(0)) <= 1e-5
    scale = float((dz_ref * (ypre - bias)).abs().reshape(groups, -1).sum(1).max())      # cancellation-free magnitude
    assert float((zw.cpu() - zw_ref).abs().max()) <= 2e-6 * scale


def test_spectral_norm_grouped_deferred_matches_two_calls():
    """Two batched reference calls through one SN conv (per-group 1/sigma, per-group weight-gradient correction with
    the coefficients from mtd_act_bwd_sn, deferred batched finishing) == two separate torch spectral-norm calls."""
    import torch.nn as nn
    from mtdgan_b200 import networks as NW, ops
    from mtdgan_b200._ext import call, fptr, ptr, stream
    torch.manual_seed(5)
    ref = nn.utils.spectral_norm(nn.Conv2d(32, 64, 3, 1, 1)).double().train()
    sd0 = {k: v.clone() for k, v in ref.state_dict().items()}
    xa, xb = _rand(3, 32, 8, 8, seed=6), _rand(3, 32, 8, 8, seed=7)
    ga, gb = _rand(3, 64, 8, 8, seed=8), _rand(3, 64, 8, 8, seed=9)
    ya = F.leaky_relu(ref(xa), 0.2)
    yb = F.leaky_relu(ref(xb), 0.2)                  # second call: second power iteration
    ((ya * ga).sum() + (yb * gb).sum()).backward()
    holder = nn.Module()
    holder.conv = nn.utils.spectral_norm(nn.Conv2d(32, 64, 3, 1, 1))
    holder.conv.load_state_dict({k: v.float() for k, v in sd0.items()})
    holder.to(DEV)
    st = NW._SNState([holder.conv], torch.device(DEV))
    u_snap = torch.empty(2, st.u_total, device=DEV)
    v_snap = torch.empty(2, st.v_total, device=DEV)
    inv = torch.empty(2, 1, device=DEV)
    for g in range(2):
        call("mtd_sn_power_iter", ptr(st.tab), 1, ptr(st.wtu), st.n_wtu, ptr(st.wv), st.n_wv, fptr(st.t_ws), st.t_elems,
             fptr(st.s_ws), fptr(u_snap[g]), fptr(v_snap[g]), fptr(inv[g]), 1, 1e-12, stream())
    xc = nhwc(torch.cat([xa, xb]).float()).to(DEV)
    cfg = ops.ConvCfg(cin=32, cout=64, pre_act=ops.ACT_LEAKY)
    w, b = holder.conv.weight_orig, holder.conv.bias
    y = ops.conv(xc, w, b, cfg, inv_sigma=inv.reshape(2), u=u_snap, v=v_snap)
    assert rel_err(nchw(y), torch.cat([ya, yb])) <= TOL
    loss = (y * nhwc(torch.cat([ga, gb]).float()).to(DEV)).sum()
    with ops.deferred_wgrad_finish():
        dw, db = torch.autograd.grad(loss, [w, b])
    torch.cuda.synchronize()
    assert rel_err(db, ref.bias.grad) <= TOL
    assert rel_err(dw, ref.weight_orig.grad) <= 2e-3        # weight gradient GEMM runs in plain TF32 on this shape
    ops.set_conv_mode("simt")
    try:
        y = ops.conv(xc, w, b, cfg, inv_sigma=inv.reshape(2), u=u_snap, v=v_snap)
        loss = (y * nhwc(torch.cat([ga, gb]).float()).to(DEV)).sum()
        with ops.deferred_wgrad_finish():
            dw, db = torch.autograd.grad(loss, [w, b])
        assert rel_err(dw, ref.weight_orig.grad) <= 2e-5    # exact-fp32 kernels
    finally:
        ops.set_conv_mode("auto", 3)


def test_repack_stale_rebuilds_all_packs_in_batches():
    """ops.repack_stale(): after in-place weight updates every registered packed copy (SIMT / tensor-core, forward /
    dgrad, stride-2 class packs) is rebuilt by the batched pack kernel and gives the same results as lazy packing."""
    from mtdgan_b200 import ops, _ext
    torch.manual_seed(11)
    layers = []
    for (cin, cout, k, s, p) in [(32, 64, 3, 1, 1), (64, 64, 4, 2, 1), (1, 32, 3, 1, 1), (64, 32, 1, 1, 0)] * 8:     # 32 layers > one batch
        w = (torch.randn(cout, cin, k, k, device=DEV) / (cin * k * k) ** 0.5).requires_grad_(True)
        b = torch.zeros(cout, device=DEV, requires_grad=True)
        layers.append((w, b, ops.ConvCfg(cin=cin, cout=cout, kh=k, kw=k, stride=s, pad=p, pre_act=ops.ACT_LEAKY)))

    def run():
        outs = []
        for w, b, cfg in layers:
            x = torch.randn(4, 16, 16, cfg.cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(cfg.cin)).requires_grad_(True)
            y = ops.conv(x, w, b, cfg)
            (gx,) = torch.autograd.grad(y.sum(), [x])
            outs.append((y.detach(), gx))
        return outs

    run()                                                     # registers fwd + dgrad packs of every layer
    with torch.no_grad():
        for w, _, _ in layers:
            w.mul_(1.5).add_(0.01)                            # bumps the version counters
    l0 = _ext.kernel_launch_count()
    n = ops.repack_stale()
    launches = _ext.kernel_launch_count() - l0
    recs = n + 3 * 8                                          # each of the 8 stride-2 dgrad packs is four class sub-packs
    assert n == 2 * len(layers) and launches == -(-recs // 24), (n, launches)
    l1 = _ext.kernel_launch_count()
    got = run()
    ops.clear_pack_cache()                                    # force lazy per-layer packing for the reference run
    want = run()
    for (y1, g1), (y2, g2) in zip(got, want):
        assert torch.equal(y1, y2) and torch.equal(g1, g2)
    assert ops.repack_stale() == 0


@pytest.mark.parametrize("passes", [1, 3], ids=["tf32", "tf32x3"])
def test_halo_tile_kernel_equals_general_kernel(passes):
    """32 -> 32 channel 3x3 layers: the halo-tile kernel (resident weights, one halo box per tile, taps as descriptor
    offsets) and the general tap-streaming kernel evaluate the same products, so forward and data gradient agree to
    summation order."""
    from mtdgan_b200 import _ext, ops
    ops.set_conv_mode("auto", passes)
    lib = _ext.load()
    try:
        x = nhwc(_rand(4, 32, 64, 64, seed=1).float()).to(DEV).requires_grad_(True)
        w = _rand(32, 32, 3, 3, seed=2, scale=1.0 / math.sqrt(288)).float().to(DEV).requires_grad_(True)
        b = _rand(32, seed=3, scale=0.1).float().to(DEV).requires_grad_(True)
        g = nhwc(_rand(4, 32, 64, 64, seed=5).float()).to(DEV)
        cfg = ops.ConvCfg(cin=32, cout=32, kh=3, kw=3, stride=1, pad=1, pre_act=ops.ACT_RELU)
        res = []
        for enabled in (1, 0):
            prev = lib.mtd_tc_set_c32(enabled)
            try:
                y = ops.conv(x, w, b, cfg)
                dx, = torch.autograd.grad(y, [x], g)
                res.append((y.detach().clone(), dx.clone()))
            finally:
                lib.mtd_tc_set_c32(prev)
        torch.cuda.synchronize()
        # same products, different accumulation order (the halo kernel keeps the small cross terms in their own accumulator)
        assert rel_err(res[0][0], res[1][0]) <= (5e-6 if passes == 3 else 2e-5)
        assert rel_err(res[0][1], res[1][1]) <= (5e-6 if passes == 3 else 2e-5)
    finally:
        ops.set_conv_mode("auto", 3)



HALO_EQ_CASES = [
    # B, H, W, C1, C2, N
    (4, 64, 64, 64, 0, 64),
    (20, 32, 32, 128, 0, 128),
    (20, 16, 16, 256, 0, 256),
    (20, 32, 32, 64, 64, 128),
    (20, 16, 16, 512, 0, 256),
    (2, 16, 8, 64, 0, 32),
]


@pytest.mark.parametrize("passes", [1, 3], ids=["tf32", "tf32x3"])
@pytest.mark.parametrize("case", HALO_EQ_CASES, ids=lambda c: "x".join(map(str, c)))
def test_streamed_halo_kernel_equals_tap_streaming_kernel(case, passes):
    """3x3 / stride-1 layers with more than 32 channels: the streamed-weight halo-tile kernel and the tap-streaming kernel
    evaluate the same error-compensated products; they differ in summation order (chunk-major k order) and, in 3xTF32
    mode, in how the activation is split (halo: hi = nearest, tap streaming: hi = the tensor core's own truncation; both
    keep hi + lo within 2^-21 of the value).  Forward and both data gradients of a two-source layer."""
    from mtdgan_b200 import _ext, ops
    B, H, W, C1, C2, N = case
    C = C1 + C2
    ops.set_conv_mode("auto", passes)
    lib = _ext.load()
    try:
        xc = nhwc(_rand(B, C, H, W, seed=21).float()).to(DEV)
        x1 = xc[..., :C1].contiguous().requires_grad_(True)
        x2 = xc[..., C1:].contiguous().requires_grad_(True) if C2 else None
        w = _rand(N, C, 3, 3, seed=22, scale=1.0 / math.sqrt(9 * C)).float().to(DEV).requires_grad_(True)
        b = _rand(N, seed=23, scale=0.1).float().to(DEV).requires_grad_(True)
        g = nhwc(_rand(B, N, H, W, seed=25).float()).to(DEV)
        # no activation: the data gradient's input must be the SAME tensor for both kernels (with one, an output within
        # rounding of zero flips its mask between the two summation orders and changes a 3 x 3 patch of dx by O(1))
        cfg = ops.ConvCfg(cin=C, cout=N, kh=3, kw=3, stride=1, pad=1, pre_act=ops.ACT_NONE)
        res = []
        for enabled in (1, 0):
            prev = lib.mtd_tc_set_halo(enabled)
            try:
                y = ops.conv(x1, w, b, cfg, x2=x2)
                grads = torch.autograd.grad(y, [x1] + ([x2] if C2 else []), g)
                res.append([y.detach().clone()] + [t.clone() for t in grads])
            finally:
                lib.mtd_tc_set_halo(prev)
        torch.cuda.synchronize()
        tol = 3e-5        # each kernel is within 5e-5 of fp64 (3xTF32) / shares the operand rounding (plain TF32)
        for got, ref in zip(res[0], res[1]):
            assert rel_err(got, ref) <= tol
    finally:
        ops.set_conv_mode("auto", 3)
