"""Data edge (SURVEY §8f-4): the GPU `window_patch` sampler against the numpy restatement of the reference's MONAI
transform chain (create_datasets/Mayo.py:117-136), BIT-EXACT (byte / index work), and the checkpoint round trip in the
reference's checkpoint layout (train.py:146-159, 276-288)."""
import io
import random

import numpy as np
import pytest
import torch

from oracle import data_edge as DE


def fake_hu(S, H, W, seed, box=None):
    """Synthetic int16 HU slice pairs: air (-1000) outside a body box, tissue values inside; the low-dose slice is the
    full-dose one plus noise.  box = (y0, y1, x0, x1) of the body."""
    rng = np.random.RandomState(seed)
    hi = np.full((S, H, W), -1000, dtype=np.int16)
    for s in range(S):
        y0, y1, x0, x1 = box if box is not None else (rng.randint(0, H // 4), H - rng.randint(1, H // 4), rng.randint(0, W // 4),
                                                     W - rng.randint(1, W // 4))
        hi[s, y0:y1, x0:x1] = rng.randint(-300, 400, size=(y1 - y0, x1 - x0)).astype(np.int16)
    lo = (hi.astype(np.int32) + rng.randint(-40, 41, size=hi.shape)).clip(-1024, 3071).astype(np.int16)
    return lo, hi


def test_window_arithmetic_is_float32_torch():
    """scale_intensity_range == the torch-CPU float32 expression MONAI 1.3.2 evaluates; values of interest are exact."""
    hu = np.arange(-1024, 3072, dtype=np.int16)
    got = DE.scale_intensity_range(hu)
    want = torch.clamp((torch.from_numpy(hu).to(torch.float32) + 160.0) / 400.0, 0, 1).numpy()
    assert got.dtype == np.float32 and np.array_equal(got, want)
    assert got[hu == -160][0] == 0.0 and got[hu == 240][0] == 1.0 and got[hu == 40][0] == 0.5


def test_product_and_oracle_draw_the_same_decisions():
    from mtdgan_b200.data import draw_decisions
    for size in ((300, 412), (64, 200), (64, 64), (70, 64)):
        a = draw_decisions(size, 64, 8, np.random.RandomState(5))
        b = DE.draw_decisions(size, 64, 8, np.random.RandomState(5))
        assert a == b
        assert all(0 <= oy <= size[0] - 64 and 0 <= ox <= size[1] - 64 for oy, ox, _, _ in a)


def test_pipeline_shapes_padding_and_empty_slice():
    lo, hi = fake_hu(1, 128, 128, 0, box=(50, 80, 40, 110))          # 30 x 70 body: padded to 64 rows
    x, y, dec = DE.window_patch_pipeline(lo[0], hi[0], np.random.RandomState(1))
    assert x.shape == (8, 1, 64, 64) and all(oy == 0 for oy, _, _, _ in dec)
    lo0 = np.full((128, 128), -1000, np.int16)
    x, y, _ = DE.window_patch_pipeline(lo0, lo0, np.random.RandomState(1))
    assert not x.any() and not y.any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["body", "small_box", "forced_aug", "empty"])
def test_gpu_sampler_bit_exact_vs_oracle(case):
    from mtdgan_b200.data import WindowPatchSampler, window_slices
    S, H, W = 6, 512, 512
    box = {"small_box": (200, 240, 100, 130), "empty": (0, 0, 0, 0)}.get(case)
    lo, hi = fake_hu(S, H, W, 11, box=box)
    kw = dict(prob_rot90=1.0, prob_flip=1.0) if case == "forced_aug" else {}
    sampler = WindowPatchSampler(seed=123, **kw)
    x, y = sampler(torch.from_numpy(lo).cuda(), torch.from_numpy(hi).cuda())
    assert x.shape == (S * 8, 1, 64, 64) and x.dtype == torch.float32
    rng = np.random.RandomState(123)
    xs, ys = [], []
    for s in range(S):
        if case == "forced_aug":        # same draws, coins forced: restate through the oracle's building blocks
            wl, wh = DE.scale_intensity_range(lo[s]), DE.scale_intensity_range(hi[s])
            y0, y1, x0, x1 = DE.foreground_bbox(wh)
            wl, wh = wl[y0:y1, x0:x1], wh[y0:y1, x0:x1]
            dec = DE.draw_decisions(wl.shape, 64, 8, rng, 1.0, 1.0)
            for oy, ox, k, f in dec:
                for src, dst in ((wl, xs), (wh, ys)):
                    p = np.flip(np.rot90(src[oy:oy + 64, ox:ox + 64], k), (0, 1))
                    dst.append(np.ascontiguousarray(p)[None])
        else:
            a, b, dec = DE.window_patch_pipeline(lo[s], hi[s], rng)
            xs += list(a); ys += list(b)
        assert dec == sampler.last_decisions[s]
    want_x, want_y = np.stack(xs), np.stack(ys)
    assert np.array_equal(x.cpu().numpy().view(np.uint32), want_x.astype(np.float32).view(np.uint32))      # bit-exact
    assert np.array_equal(y.cpu().numpy().view(np.uint32), want_y.astype(np.float32).view(np.uint32))
    full = window_slices(torch.from_numpy(hi).cuda())
    assert np.array_equal(full.cpu().numpy()[:, 0].view(np.uint32), DE.scale_intensity_range(hi).view(np.uint32))


def test_cpu_tensors_rejected():
    from mtdgan_b200.data import WindowPatchSampler
    from mtdgan_b200._ext import MtdError
    with pytest.raises(MtdError):
        WindowPatchSampler()(torch.zeros(1, 64, 64, dtype=torch.int16), torch.zeros(1, 64, 64, dtype=torch.int16))


# ---- checkpoint round trip -------------------------------------------------------------------------------------
def test_checkpoint_self_round_trip_cpu():
    """state_dict / optimizer state written by the drop-in loads back bit-for-bit (keys of train.py:279-287)."""
    from arch.Ours.networks import Ablation_CLS
    from mtdgan_b200 import checkpoint as CK
    torch.manual_seed(0)
    m = Ablation_CLS()
    oD = torch.optim.AdamW(m.Discriminator.parameters(), lr=1e-4)
    oG = torch.optim.AdamW(m.Generator.parameters(), lr=1e-4)
    buf = io.BytesIO()
    torch.save(CK.checkpoint_dict(m, oD, None, oG, None, epoch=7), buf)
    buf.seek(0)
    ck = torch.load(buf, map_location="cpu", weights_only=False)
    assert tuple(ck.keys()) == CK.KEYS
    torch.manual_seed(1)
    m2 = Ablation_CLS()
    assert CK.load_checkpoint(ck, m2) == 8
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_checkpoint_in_reference_layout_loads_and_returns():
    """A checkpoint as the reference's train.py writes it (the model's state_dict under the reference's 326 keys, pinned
    by its init fingerprint state_summary.pt; torch.optim.AdamW state after one optimizer step; dict layout of
    train.py:279-287, with DataParallel-style '.module' keys to exercise :149) loads into the drop-in model and the fused
    optimizer, and a checkpoint the drop-in writes loads back into a model and torch.optim.AdamW — all tensors equal."""
    from _golden_util import load
    from arch.Ours.networks import MTD_GAN_Method
    from mtdgan_b200 import checkpoint as CK
    from mtdgan_b200.optim import FusedAdamW
    torch.manual_seed(3); random.seed(3)
    rm = MTD_GAN_Method()
    assert list(rm.state_dict().keys()) == list(load("state_summary.pt").keys())
    rD = torch.optim.AdamW([{"params": list(rm.Discriminator.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
    rG = torch.optim.AdamW(rm.Generator.parameters(), lr=1e-4, weight_decay=5e-4)
    g = torch.Generator().manual_seed(2)
    for p in rm.parameters():                               # seeded gradients (the drop-in has no CPU forward): one step each
        p.grad = 1e-3 * torch.randn(p.shape, generator=g)
    rD.step(); rG.step()
    sch = torch.optim.lr_scheduler.LambdaLR(rG, lambda e: 0.5)
    ck = {"model_state_dict": {k.replace("Generator.", "Generator.module.", 1) if k.startswith("Generator.encoder.0") else k: v
                               for k, v in rm.state_dict().items()},
          "optimizer_D": rD.state_dict(), "scheduler_D": None, "optimizer_G": rG.state_dict(), "scheduler_G": sch.state_dict(),
          "epoch": 4, "args": None}
    mine = MTD_GAN_Method()
    mD = FusedAdamW([{"params": list(mine.Discriminator.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
    mG = FusedAdamW(mine.Generator.parameters(), lr=1e-4, weight_decay=5e-4)
    assert CK.load_checkpoint(ck, mine, mD, None, mG, None) == 5
    for (k, a), (k2, b) in zip(rm.state_dict().items(), mine.state_dict().items()):
        assert k == k2 and torch.equal(a, b), k
    for rp, mp in zip(rm.Generator.parameters(), mine.Generator.parameters()):
        for key in ("step", "exp_avg", "exp_avg_sq"):
            assert torch.equal(torch.as_tensor(rG.state[rp][key]).float(), torch.as_tensor(mG.state[mp][key]).float().cpu()), key
    # and back: what the drop-in writes, a fresh model and torch.optim.AdamW load
    back = CK.checkpoint_dict(mine, mD, None, mG, None, epoch=5)
    rm2 = MTD_GAN_Method()
    rm2.load_state_dict(back["model_state_dict"])
    rG2 = torch.optim.AdamW(rm2.Generator.parameters(), lr=1e-4, weight_decay=5e-4)
    rG2.load_state_dict(back["optimizer_G"])
    for (k, a), (_, b) in zip(rm.state_dict().items(), rm2.state_dict().items()):
        assert torch.equal(a, b), k
    for rp, rp2 in zip(rm.Generator.parameters(), rm2.Generator.parameters()):
        for key in ("step", "exp_avg", "exp_avg_sq"):
            assert torch.equal(torch.as_tensor(rG.state[rp][key]).float(), torch.as_tensor(rG2.state[rp2][key]).float()), key
