"""The Res-FFT-Conv frequency branch at every H, W in [1, 512] (the reference's torch.fft.rfft2 takes any size).
Lengths 64, 128, 256, 512 run the four-step FFTs; every other length runs the Bluestein kernels.  Checked against
torch.fft in fp64 and against the CPU oracle.  test_fft_dispatch.py checks that the FFT tests together reach every
kernel instance of either class."""
import random

import pytest
import torch

from _golden_util import rel_err
from oracle import mtdgan_oracle as O

DEV = "cuda"
gpu = pytest.mark.gpu

ROW_LENGTHS = [1, 2, 7, 37, 63, 65, 96, 100, 255, 384, 500, 509, 511]
# (128, 128) and (256, 256) run the four-step columns at H = 128 and 256; (64, 7) and (7, 64) mix the four-step and
# Bluestein classes in one block
BLOCK_SIZES = [(1, 1), (7, 5), (63, 65), (96, 100), (37, 509), (509, 37), (300, 300), (384, 512), (512, 384), (511, 509),
               (128, 128), (256, 256), (64, 7), (7, 64)]


class Tol:
    """Per-mode output tolerances of test_gpu_model.py (norm-wise relative errors)."""
    def __init__(self, mode):
        self.mode = mode
        self.out = {"simt": 1e-4, "tc3": 3e-4, "tc1": 1e-2}[mode]


@pytest.fixture(params=["simt", "tc3", "tc1"])
def conv_mode(request):
    from mtdgan_b200 import ops
    if request.param == "simt":
        ops.set_conv_mode("simt")
    else:
        ops.set_conv_mode("auto", 3 if request.param == "tc3" else 1)
    yield Tol(request.param)
    ops.set_conv_mode("auto", 3)


def seeded_model():
    from arch.Ours.networks import MTD_GAN_Method
    torch.manual_seed(2024)
    random.seed(2024)
    return MTD_GAN_Method().to(DEV)


def slices(n, H, W, seed):
    """synthetic_pair's noisy input at any H x W: plateaus at 0 and 1 like HU windowing."""
    g = torch.Generator().manual_seed(seed)
    y = torch.clamp(1.6 * torch.rand(n, 1, H, W, generator=g) - 0.3, 0, 1)
    return torch.clamp(y + 0.1 * torch.randn(n, 1, H, W, generator=g), 0, 1)


_ORACLE = {}


def oracle_generator(sd, x, key):
    if key not in _ORACLE:
        with torch.no_grad():
            _ORACLE[key] = torch.cat([O.generator_forward(sd, x[i:i + 1]) for i in range(x.shape[0])])
    return _ORACLE[key]


def test_supported_geometry():
    from mtdgan_b200 import _ext
    lib = _ext.load()
    assert all(lib.mtd_fft_supported(h, w, 32) == 1 for h in range(1, 513) for w in range(1, 513))
    for h, w in [(0, 64), (64, 0), (513, 64), (64, 513), (513, 513)]:
        assert lib.mtd_fft_supported(h, w, 32) == 0, (h, w)
    assert lib.mtd_fft_supported(64, 64, 16) == 0 and lib.mtd_fft_supported(64, 64, 64) == 0


@gpu
@pytest.mark.parametrize("H", [1, 6, 33])
@pytest.mark.parametrize("W", ROW_LENGTHS)
def test_rows_any_length(H, W):
    """Half spectrum against torch.fft.rfft(norm="ortho") in fp64, and irfft_W(rfft_W(x)) == x."""
    from mtdgan_b200._ext import call, fptr, stream, load as libload
    B, C = 2, 32
    x = torch.randn(B, H, W, C, generator=torch.Generator().manual_seed(W * 1000 + H)).to(DEV)
    spec = torch.empty(libload().mtd_fft_spec_elems(B, H, W, C), device=DEV)
    call("mtd_fft_rows_fwd", fptr(x), fptr(spec), B, H, W, C, stream())
    back = torch.empty_like(x)
    call("mtd_fft_rows_inv", fptr(spec), None, None, fptr(back), B, H, W, C, stream())
    want = torch.fft.rfft(x.double().cpu(), dim=2, norm="ortho")            # (B,H,Wh,C)
    got = torch.view_as_complex(spec.view(B, W // 2 + 1, H, C, 2)).permute(0, 2, 1, 3).cpu()
    fwd = float((got - want).abs().max() / want.abs().max())
    inv = rel_err(back, x)
    print("rows W=%d H=%d: rfft err %.2e, roundtrip err %.2e" % (W, H, fwd, inv))
    assert fwd <= 1e-5 and inv <= 1e-5


@gpu
@pytest.mark.parametrize("grad", [False, True], ids=["no_grad", "grad"])
@pytest.mark.parametrize("mode", ["simt", "auto"])
@pytest.mark.parametrize("H,W", BLOCK_SIZES)
def test_fft_block_any_size_vs_oracle(H, W, mode, grad):
    """FFT_ConvBlock forward against the fp64 oracle, in the inference form (no autograd graph: the identity branch rides
    in the conv epilogue) and the training form (spectrum saved for backward, out-of-place mix)."""
    from arch.Ours.networks import FFT_ConvBlock
    from mtdgan_b200 import ops
    torch.manual_seed(5)
    blk = FFT_ConvBlock(32).to(DEV)
    x = 0.5 * torch.randn(1, 32, H, W, generator=torch.Generator().manual_seed(H * 1000 + W))
    ops.set_conv_mode(mode, 3 if mode == "auto" else None)
    try:
        if grad:
            out = blk(x.to(DEV).requires_grad_(True))
        else:
            with torch.no_grad():
                out = blk(x.to(DEV))
        torch.cuda.synchronize()
    finally:
        ops.set_conv_mode("auto", 3)
    p = {k: v.detach().double().cpu() for k, v in blk.named_parameters()}
    want = O.fft_conv_block(x.double(), p["img_conv.weight"], p["img_conv.bias"], p["fft_conv.weight"], p["fft_conv.bias"])
    err = rel_err(out, want)
    print("FFT block %dx%d (%s, %s): rel err %.2e" % (H, W, mode, "grad" if grad else "no_grad", err))
    assert err <= 1e-4


@gpu
@pytest.mark.parametrize("B,H,W", [(2, 96, 100), (1, 500, 509)])
def test_generator_any_size_vs_oracle(B, H, W, conv_mode):
    m = seeded_model().eval()
    x = slices(B, H, W, seed=H + W)
    sd = {k: v.detach().cpu() for k, v in m.Generator.state_dict().items()}
    want = oracle_generator(sd, x, (B, H, W))
    with torch.no_grad():
        out = m.Generator(x.to(DEV))
    assert out.shape == (B, 1, H, W) and float(out.min()) >= 0.0
    err = rel_err(out, want)
    print("generator %dx%dx%d forward (%s): rel err %.2e" % (B, H, W, conv_mode.mode, err))
    assert err <= conv_mode.out


@gpu
def test_graphed_generator_any_size():
    """Three 509 x 384 slices through the CUDA-graph runner at micro-batch 2 (the second replay's tail is zero padded)."""
    from mtdgan_b200.inference import GraphedGenerator
    m = seeded_model().eval()
    x = slices(3, 509, 384, seed=41)
    sd = {k: v.detach().cpu() for k, v in m.Generator.state_dict().items()}
    want = oracle_generator(sd, x, (3, 509, 384))
    runner = GraphedGenerator(m.Generator, 509, 384, micro_batch=2).capture()
    got = runner(x.to(DEV))
    torch.cuda.synchronize()
    errs = [rel_err(got[i], want[i]) for i in range(3)]
    print("graphed 509x384 inference: per-slice rel err", ["%.2e" % e for e in errs])
    assert max(errs) <= Tol("tc3").out


@gpu
def test_out_of_range_and_backward_raise():
    from arch.Ours.networks import FFT_ConvBlock
    from mtdgan_b200 import _ext
    blk = FFT_ConvBlock(32).to(DEV)
    with pytest.raises(_ext.MtdError, match=r"1 <= H, W <= 512"):
        with torch.no_grad():
            blk(torch.zeros(1, 32, 513, 64, device=DEV))
    # (512, 64): power-of-two, but the backward kernel's two column slices at H = 512 exceed shared memory
    for H, W in [(96, 100), (512, 64)]:
        x = torch.randn(1, 32, H, W, device=DEV, requires_grad=True)
        out = blk(x)
        with pytest.raises(_ext.MtdError, match=r"backward is built for"):
            out.sum().backward()
    torch.cuda.synchronize()
