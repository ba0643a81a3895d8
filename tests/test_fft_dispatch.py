"""Every kernel instance of the Res-FFT-Conv frequency branch (csrc/fft_block.cu) against fp64, and the FFT block's
backward at every size it admits.

The host code picks a kernel instance by transform length: the four-step FFTs at 64, 128, 256 and 512, Bluestein at
every other length, with one instance per convolution length M = max(64, next power of two >= 2N - 1).  Thread
mapping, row packing, the channel-mix work split and the shared-memory layout change with the instance, so an instance
no test runs can be wrong while the suite passes.  The dispatch is restated below; test_fft_tests_reach_every_instance
checks that the size lists of the FFT tests reach every instance, and test_dispatch_restatement_matches_source that
the restatement still matches the sources, so adding an instance or dropping a size fails without a GPU.

References are fp64 on the CPU; errors are max |a - b| / max |b|."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

import test_fft_any_size
import test_gpu_kernels
from _golden_util import rel_err
from oracle import mtdgan_oracle as O

DEV = "cuda"
gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ---- the host dispatch, restated -------------------------------------------------------------------------------------
FOUR_STEP = {64: (8, 8), 128: (8, 16), 256: (16, 16), 512: (16, 32)}              # length -> (N1, N2)
BLUESTEIN = {64: (8, 8), 128: (8, 16), 256: (16, 16), 512: (16, 32), 1024: (32, 32)}   # M -> (N1, N2)


def fft_len_ok(n):
    return n in FOUR_STEP


def blue_len(n):
    m = 64
    while m < 2 * n - 1:
        m <<= 1
    return m


def rows_per_cta(w):
    """RowsCfg<N1, N2>::RPB of the four-step row kernels."""
    n1, n2 = FOUR_STEP[w]
    return 2 if 16 * n2 <= 128 and 16 * n1 <= 128 else 1


def backward_ok(h, w):
    return fft_len_ok(h) and h <= 256 and fft_len_ok(w)


def instance(n):
    return ("four-step", n) if fft_len_ok(n) else ("Bluestein M", blue_len(n))


# ---- size lists of the tests in this file ----------------------------------------------------------------------------
ROWS_INV_LENGTHS = [64, 128, 256, 512, 100, 509]                   # + one even and one odd Bluestein length
COL_HEIGHTS = [64, 128, 256, 512, 1, 32, 33, 65, 129, 255, 257, 511]   # four-step, then the Bluestein class boundaries
BWD_CASES = [(5 if (h, w) == (64, 512) else 2, h, w) for h in (64, 128, 256) for w in (64, 128, 256, 512)]


def _read(rel):
    with open(os.path.join(ROOT, rel)) as fh:
        return fh.read()


def _dispatch_cases(src, macro):
    body = re.search(r"#define %s\(.*?\)(.*?)default:" % macro, src, re.S).group(1)
    return {int(n): (int(a), int(b)) for n, a, b in re.findall(r"case (\d+): \{ CALL\((\d+), (\d+)\)", body)}


def test_dispatch_restatement_matches_source():
    src = re.sub(r"\s+", " ", _read("mtd-gan_b200/csrc/fft_block.cu"))
    assert _dispatch_cases(src, "MTD_FFT_DISPATCH") == FOUR_STEP
    assert _dispatch_cases(src, "MTD_BLUE_DISPATCH") == BLUESTEIN
    assert {int(n) for n in re.findall(r"n == (\d+)", re.search(r"bool fft_len_ok\(int n\) \{(.*?)\}", src).group(1))} \
        == set(FOUR_STEP)
    assert "int blue_len(int n) { int m = 64; while (m < 2 * n - 1) m <<= 1; return m; }" in src
    assert {blue_len(n) for n in range(1, 513) if not fft_len_ok(n)} == set(BLUESTEIN)
    assert "static constexpr int IA = kQ * N2;" in src and "static constexpr int IB = kQ * N1;" in src
    assert "static constexpr int RPB = (IA <= 128 && IB <= 128) ? 2 : 1;" in src
    assert "fft_len_ok(H) && H <= 256 && fft_len_ok(W)" in src                  # mtd_fft_cols_mix_bwd
    hs, ws = re.search(r"if H not in \(([\d, ]+)\) or W not in \(([\d, ]+)\):", _read("mtd-gan_b200/ops.py")).groups()
    admitted = {(h, w) for h in range(1, 513) for w in range(1, 513) if backward_ok(h, w)}
    assert {(int(h), int(w)) for h in hs.split(",") for w in ws.split(",")} == admitted       # FFTConvBlockFn.backward


def test_fft_tests_reach_every_instance():
    missing = []

    def need(what, have, want):
        missing.extend("%s: %s" % (what, w) for w in sorted(set(want) - set(have)))

    row_cases = test_gpu_kernels.FFT_ROW_CASES
    need("rows four-step W (test_gpu_kernels.FFT_ROW_CASES)", [w for _, _, w in row_cases], FOUR_STEP)
    need("rows four-step W with a half-filled last CTA: odd B*H (test_gpu_kernels.FFT_ROW_CASES)",
         [w for b, h, w in row_cases if fft_len_ok(w) and (b * h) % rows_per_cta(w)],
         [w for w in FOUR_STEP if rows_per_cta(w) > 1])
    need("rows Bluestein M (test_fft_any_size.ROW_LENGTHS)",
         [blue_len(w) for w in test_fft_any_size.ROW_LENGTHS if not fft_len_ok(w)], BLUESTEIN)
    need("rows inverse four-step W (ROWS_INV_LENGTHS)", ROWS_INV_LENGTHS, FOUR_STEP)
    need("rows inverse Bluestein W parity (ROWS_INV_LENGTHS)",
         ["odd" if w % 2 else "even" for w in ROWS_INV_LENGTHS if not fft_len_ok(w)], ["even", "odd"])
    need("columns + mix (COL_HEIGHTS)", [instance(h) for h in COL_HEIGHTS],
         [("four-step", n) for n in FOUR_STEP] + [("Bluestein M", m) for m in BLUESTEIN])
    need("columns four-step H in a block (test_fft_any_size.BLOCK_SIZES)",
         [h for h, _ in test_fft_any_size.BLOCK_SIZES], FOUR_STEP)
    need("backward (H, W) (BWD_CASES)", [(h, w) for _, h, w in BWD_CASES],
         [(h, w) for h in FOUR_STEP for w in FOUR_STEP if backward_ok(h, w)])
    assert not missing, "FFT kernel instances no test reaches:\n  " + "\n  ".join(missing)
    assert all(backward_ok(h, w) for _, h, w in BWD_CASES)


# ---- rows inverse ----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("W", ROWS_INV_LENGTHS)
def test_rows_inv_vs_irfft(W):
    """mtd_fft_rows_inv with both residual adds on a random half spectrum whose DC and Nyquist columns carry imaginary
    parts.  irfft ignores those parts; an odd W has no Nyquist column, so its last column's imaginary part counts."""
    from mtdgan_b200._ext import call, fptr, stream
    B, H, C = 3, 5, 32                                  # 15 rows: odd, so the two-row CTAs of W = 64 end half filled
    g = torch.Generator().manual_seed(W)
    spec = torch.randn(B, W // 2 + 1, H, C, 2, generator=g)
    add1, add2 = torch.randn(B, H, W, C, generator=g), torch.randn(B, H, W, C, generator=g)
    dev = [t.to(DEV) for t in (spec, add1, add2)]                 # held: the kernel runs after fptr() returns
    out = torch.empty(B, H, W, C, device=DEV)
    call("mtd_fft_rows_inv", *map(fptr, dev), fptr(out), B, H, W, C, stream())
    fft = torch.fft.irfft(torch.view_as_complex(spec.double()).permute(0, 2, 1, 3), n=W, dim=2, norm="ortho")
    err = float((out.double().cpu() - (fft + add1.double() + add2.double())).abs().max() / fft.abs().max())
    print("rows inverse W=%d: err %.2e" % (W, err))
    assert err <= 1e-5


# ---- columns + channel mix -------------------------------------------------------------------------------------------
def cols_mix_ref(spec, w, b):
    """spec (S, H, 32) complex128 -> ifft_H(complex(chunk(relu(conv1x1(cat[Re, Im](fft_H(spec))))))), ortho."""
    f = torch.fft.fft(spec, dim=1, norm="ortho")
    y = torch.relu(torch.cat([f.real, f.imag], -1) @ w.t() + b)
    re, im = y.chunk(2, -1)
    return torch.fft.ifft(torch.complex(re, im), dim=1, norm="ortho")


@gpu
@pytest.mark.parametrize("inplace", [False, True], ids=["out_of_place", "in_place"])
@pytest.mark.parametrize("H", COL_HEIGHTS)
def test_cols_mix_vs_fp64(H, inplace):
    """mtd_fft_cols_mix on a random spectrum of B * (W/2 + 1) = 6 column slices.  In place (spec_in == spec_out) is the
    inference form; out of place the training form."""
    from mtdgan_b200._ext import call, fptr, stream
    B, W, C = 2, 4, 32
    S = B * (W // 2 + 1)
    spec = torch.randn(S, H, C, 2, generator=torch.Generator().manual_seed(H))
    torch.manual_seed(H)
    conv = torch.nn.Conv2d(2 * C, 2 * C, 1)                 # fft_conv at its default initialisation
    w, b = conv.weight.detach().view(2 * C, 2 * C), conv.bias.detach()
    src, wd, bd = spec.to(DEV), w.contiguous().to(DEV), b.to(DEV)
    dst = src if inplace else torch.empty_like(src)
    call("mtd_fft_cols_mix", fptr(src), fptr(dst), fptr(wd), fptr(bd), B, H, W, C, stream())
    want = cols_mix_ref(torch.view_as_complex(spec.double()), w.double(), b.double())
    err = rel_err(dst, torch.view_as_real(want))
    print("columns + mix H=%d (%s): err %.2e" % (H, "in place" if inplace else "out of place", err))
    assert err <= 1e-5


# ---- FFT block backward ----------------------------------------------------------------------------------------------
def margin_bias(z):
    """Per-channel bias that keeps every pre-activation z + b of a ReLU away from zero: b = -(midpoint of the widest gap
    between neighbouring values of the channel within its 20th to 80th percentile).  A pre-activation within rounding
    of zero may take either ReLU branch in any fp32 evaluation, and one flip moves a gradient sum by ~1/sqrt(count)
    (1e-3 to 3e-2 at these sizes), which would hide a real error of that size.  Returns (b as fp32, the smallest
    |z + b| over max |z + b|)."""
    v = z.transpose(0, 1).reshape(z.shape[1], -1).sort(dim=1).values
    n = v.shape[1]
    lo, hi = n // 5, 4 * n // 5
    i = (v[:, lo + 1:hi + 1] - v[:, lo:hi]).argmax(dim=1, keepdim=True) + lo
    b = (-(v.gather(1, i) + v.gather(1, i + 1)) / 2).squeeze(1).float()
    zb = z + b.double().view(1, -1, *[1] * (z.dim() - 2))
    return b, float(zb.abs().min() / zb.abs().max())


_PROBLEMS = {}


def block_problem(B, H, W, freq_only):
    """Seeded FFT_ConvBlock parameters, input, output gradient, and the oracle's fp32 and fp64 gradients.  freq_only:
    img_conv zeroed, so x.grad - dout is the frequency branch's input gradient alone."""
    key = (B, H, W, freq_only)
    if key in _PROBLEMS:
        return _PROBLEMS[key]
    from arch.Ours.networks import FFT_ConvBlock
    torch.manual_seed(5)
    blk = FFT_ConvBlock(32)
    g = torch.Generator().manual_seed(B * 1000003 + H * 1000 + W)
    x = 0.5 * torch.randn(B, 32, H, W, generator=g)
    dout = torch.randn(B, 32, H, W, generator=g)
    x64, margins = x.double(), []
    with torch.no_grad():
        if freq_only:
            blk.img_conv.weight.zero_()
            blk.img_conv.bias.zero_()
        else:
            b, m = margin_bias(F.conv2d(x64, blk.img_conv.weight.double(), padding=1))
            blk.img_conv.bias.copy_(b)
            margins.append(m)
        s = torch.fft.rfft2(x64, norm="ortho")
        b, m = margin_bias(F.conv2d(torch.cat([s.real, s.imag], 1), blk.fft_conv.weight.double()))
        blk.fft_conv.bias.copy_(b)
        margins.append(m)
    params = {k: v.detach().clone() for k, v in blk.named_parameters()}
    grads = {}
    for dt in (torch.float32, torch.float64):
        xs = x.detach().to(dt).requires_grad_(True)
        ps = {k: v.detach().to(dt).requires_grad_(True) for k, v in params.items()}
        O.fft_conv_block(xs, ps["img_conv.weight"], ps["img_conv.bias"], ps["fft_conv.weight"], ps["fft_conv.bias"]) \
            .backward(dout.to(dt))
        grads[dt] = {"dx": xs.grad, "dx - dout": xs.grad - dout.to(dt), **{k: p.grad for k, p in ps.items()}}
    _PROBLEMS[key] = (params, x, dout, grads[torch.float32], grads[torch.float64], min(margins))
    return _PROBLEMS[key]


def run_block(params, x, dout):
    from arch.Ours.networks import FFT_ConvBlock
    blk = FFT_ConvBlock(32)
    blk.load_state_dict(params)
    blk = blk.to(DEV)
    xd = x.to(DEV).requires_grad_(True)
    blk(xd).backward(dout.to(DEV))
    torch.cuda.synchronize()
    return {"dx": xd.grad, "dx - dout": xd.grad.double().cpu() - dout.double(),
            **{k: p.grad for k, p in blk.named_parameters()}}


def check_grads(what, got, g32, g64, keys, tol_of):
    """Per-tensor bound max(tol, 30 x the oracle's own fp32-vs-fp64 gap); every error is printed before any assert."""
    res = {k: (rel_err(got[k], g64[k]), max(tol_of(k), 30 * rel_err(g32[k], g64[k]))) for k in keys}
    print("%s: %s" % (what, ", ".join("%s %.2e (tol %.1e)" % (k, e, t) for k, (e, t) in res.items())))
    bad = {k: v for k, v in res.items() if v[0] > v[1]}
    assert not bad, "%s: over tolerance %s" % (what, bad)


@gpu
@pytest.mark.parametrize("mode", ["simt", "auto"])
@pytest.mark.parametrize("B,H,W", BWD_CASES)
def test_fft_block_backward_vs_fp64(B, H, W, mode):
    """FFT_ConvBlock forward + backward at every size the backward admits, all five gradients against fp64 autograd
    through the oracle.  auto: img_conv's weight gradient runs in plain TF32 on the tensor cores (2e-3)."""
    from mtdgan_b200 import ops
    params, x, dout, g32, g64, margin = block_problem(B, H, W, freq_only=False)
    assert margin > 1e-6
    ops.set_conv_mode(mode, 3 if mode == "auto" else None)
    try:
        got = run_block(params, x, dout)
    finally:
        ops.set_conv_mode("auto", 3)
    check_grads("FFT block backward %dx%dx%d (%s, ReLU margin %.1e)" % (B, H, W, mode, margin), got, g32, g64,
                ["dx", "img_conv.weight", "img_conv.bias", "fft_conv.weight", "fft_conv.bias"],
                lambda k: 2e-3 if (mode == "auto" and k == "img_conv.weight") else 1e-4)


@gpu
@pytest.mark.parametrize("B,H,W", BWD_CASES)
def test_fft_block_backward_frequency_branch(B, H, W):
    """img_conv zeroed: x.grad - dout is the frequency branch's input gradient alone, undiluted by the identity and
    image terms, and compared with the oracle's on its own."""
    params, x, dout, g32, g64, margin = block_problem(B, H, W, freq_only=True)
    assert margin > 1e-6
    got = run_block(params, x, dout)
    check_grads("FFT block frequency branch %dx%dx%d (ReLU margin %.1e)" % (B, H, W, margin), got, g32, g64,
                ["dx - dout", "fft_conv.weight", "fft_conv.bias"], lambda k: 1e-4)
