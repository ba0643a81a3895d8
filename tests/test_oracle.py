"""Pins the CPU oracle (oracle/mtdgan_oracle.py): against the golden vectors generated from the live
reference, against the reference's only known-answer vector (module/pcgrad.py demo), and against numpy
restatements of the FFT / mask contracts."""
import random

import numpy as np
import pytest
import torch

from _golden_util import check_summary, load, rel_err
from oracle import mtdgan_oracle as O

torch.set_num_threads(8)


def drop_mask(b, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, 512, generator=g) >= 0.3).float() / 0.7


@pytest.fixture(scope="module")
def seeded_sd():
    """Reference-identical initial weights: the drop-in modules reproduce the reference's RNG order
    (checked in test_boundary_cpu.py::test_init_fingerprint), so they provide the state dict."""
    from arch.Ours.networks import MTD_GAN_Method
    torch.manual_seed(2024)
    random.seed(2024)
    m = MTD_GAN_Method()
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def test_generator_forward_64_vs_golden(seeded_sd):
    x = O.synthetic_pair(2, 64, seed=11)[0]
    with torch.no_grad():
        out = O.generator_forward(seeded_sd, x, "Generator.")
    assert rel_err(out, load("gen_fwd_64.pt")["out"]) <= 1e-6


def test_fft_block_vs_golden():
    from arch.Ours.networks import FFT_ConvBlock
    torch.manual_seed(5)
    blk = FFT_ConvBlock(32)
    g = torch.Generator().manual_seed(6)
    x = (0.5 * torch.randn(1, 32, 64, 64, generator=g)).requires_grad_(True)
    wgt = torch.randn(1, 32, 64, 64, generator=g)
    p = {k: v.detach().clone().requires_grad_(True) for k, v in blk.state_dict().items()}
    out = O.fft_conv_block(x, p["img_conv.weight"], p["img_conv.bias"], p["fft_conv.weight"], p["fft_conv.bias"])
    (out * wgt).sum().backward()
    fix = load("fftblock_64.pt")
    assert rel_err(out, fix["out"]) <= 1e-6
    assert rel_err(x.grad, load("fftblock_64_dx.pt")["dx"]) <= 1e-6
    for k, g_ref in fix["grads"].items():
        assert rel_err(p[k].grad, g_ref) <= 1e-5, k


def test_discriminator_vs_golden(seeded_sd):
    sd = {k[len("Discriminator."):]: v.clone() for k, v in seeded_sd.items() if k.startswith("Discriminator.")}
    for k, v in sd.items():
        if not k.endswith(("weight_u", "weight_v")):
            v.requires_grad_(True)
    y = O.synthetic_pair(2, 64, seed=13)[1]
    enc, dec, rec = O.discriminator_forward(sd, y, True, drop_mask(2, 14))
    fix = load("disc_64.pt")
    assert rel_err(enc, fix["enc"]) <= 1e-6 and rel_err(dec, fix["dec"]) <= 1e-6 and rel_err(rec, fix["rec"]) <= 1e-6
    g = torch.Generator().manual_seed(15)
    a, b, c = torch.randn(enc.shape, generator=g), torch.randn(dec.shape, generator=g), torch.randn(rec.shape, generator=g)
    ((enc * a).sum() + (dec * b).sum() / 64 + (rec * c).sum() / 64).backward()
    for k, s in fix["grads"].items():
        check_summary(sd[k].grad, s, 1e-5, k)
    for k, s in fix["buffers"].items():
        check_summary(sd[k], s, 1e-6, k)
    with torch.no_grad():
        e2, d2, r2 = O.discriminator_forward(sd, y, False, None)
    assert rel_err(e2, fix["eval_enc"]) <= 1e-6 and rel_err(d2, fix["eval_dec"]) <= 1e-6


def test_train_step_losses_and_pcgrad_vs_golden(seeded_sd):
    fix = load("train_step_b4.pt")
    sd = {k: v.clone() for k, v in seeded_sd.items()}
    for k, v in sd.items():
        if k.startswith("Discriminator.") and not k.endswith(("weight_u", "weight_v")):
            v.requires_grad_(True)
    x, y = O.synthetic_pair(4, 64, seed=1234)
    losses, det = O.d_loss(sd, x, y, True, [drop_mask(4, 21 + i) for i in range(4)])
    assert torch.allclose(losses, fix["d_losses"], rtol=1e-5, atol=1e-12)
    for k, v in fix["d_details"].items():
        assert torch.allclose(det[k], v, rtol=1e-5, atol=1e-12), k
    shared = [sd["Discriminator." + n] for n in O.d_shared_names()]
    grads = [torch.autograd.grad(l, shared, retain_graph=True) for l in losses]
    flat = [torch.cat([t.flatten() for t in tg]).double() for tg in grads]
    gram = np.array([[float(p @ q) for q in flat] for p in flat])
    assert np.allclose(gram, fix["gram"].numpy(), rtol=1e-4, atol=1e-14)
    random.seed(99)
    merged = O.pcgrad_project_lists(list(grads), "sum")
    for n, g in zip(O.d_shared_names(), merged):
        check_summary(g, fix["d_grads"][n], 1e-4, n)
    # Gram-space restatement agrees with the vector-space loop
    random.seed(99)
    idx, orders = [0, 1, 2], []
    for _ in range(3):
        random.shuffle(idx)
        orders.append(list(idx))
    C = O.pcgrad_coefficients(gram, orders)
    w = C.sum(0)
    merged2 = sum(float(w[k]) * flat[k] for k in range(3))
    merged1 = torch.cat([g.flatten() for g in merged]).double()
    assert float((merged1 - merged2).norm() / merged1.norm()) <= 1e-5


# SURVEY §4: the reference's printed self-check (4 decimals, torch CPU)
_DEMO_PRINTED = [
    [[[-0.5955, -0.1214, 0.7084], [-0.0214, -0.3130, -0.1566], [0.5900, 0.1193, -0.7024], [0.4459, 0.0869, -0.5328]],
     [0.1312, -0.3516, -0.1312, -0.1028]],
    [[[0.1543, 0.1705, -0.1015], [-0.4761, -0.3491, 0.4177]], [0.1266, -0.1860],
     [[-0.0333, 0.0969], [-0.1064, 0.0918], [-0.0381, -0.0076], [-0.0717, 0.0192]], [-0.1726, -0.2270, -0.0211, -0.0894],
     [[0.1493, 0.0015], [-0.3189, 0.1969], [0.0228, -0.0440], [-0.1457, 0.0503]], [0.1246, -0.5640, 0.0848, -0.1987]],
]


def _demo_with(project):
    """module/pcgrad.py:165-195 with `project(grads, has_grads) -> merged flat gradient`."""
    import torch.nn as nn
    from module.pcgrad import TestNet, MultiHeadTestNet
    out = []
    for cls, heads in ((TestNet, False), (MultiHeadTestNet, True)):
        torch.manual_seed(4)
        x, y = torch.randn(2, 3), torch.randn(2, 4)
        net = cls()
        if heads:
            y1, y2 = net(x)
            objs = [nn.MSELoss()(y1, y), nn.MSELoss()(y2, y)]
        else:
            yp = net(x)
            objs = [nn.L1Loss()(yp, y), nn.MSELoss()(yp, y)]
        params = list(net.parameters())
        grads, has = [], []
        for o in objs:
            gs = torch.autograd.grad(o, params, retain_graph=True, allow_unused=True)
            grads.append(torch.cat([(torch.zeros_like(p) if g is None else g).flatten() for g, p in zip(gs, params)]))
            has.append(torch.cat([(torch.zeros_like(p) if g is None else torch.ones_like(p)).flatten()
                                  for g, p in zip(gs, params)]))
        merged = project(grads, has)
        res, off = [], 0
        for p in params:
            res.append(merged[off:off + p.numel()].view(p.shape))
            off += p.numel()
        out.append(res)
    return out


def test_pcgrad_demo_known_answer():
    got = _demo_with(lambda g, h: O.pcgrad_project_flat(g, h))
    gold = load("pcgrad_demo.pt")["grads"]
    for net_got, net_gold, net_print in zip(got, gold, _DEMO_PRINTED):
        for a, b, c in zip(net_got, net_gold, net_print):
            assert torch.allclose(a, b, rtol=1e-6, atol=1e-7)
            assert torch.allclose(a, torch.tensor(c), atol=6e-5)


def test_loss_terms_vs_golden():
    fix = load("losses.pt")
    xs, ys = O.synthetic_pair(4, 64, seed=32)
    for name, fn in (("ls_gan1", lambda p: O.ls_gan(p, 1.0)), ("nds0", lambda p: O.nds_loss(p, 0.0, xs - ys)),
                     ("charb", lambda p: O.charbonnier(p, ys)), ("edge", lambda p: O.edge_loss(p, ys))):
        p = fix["pred"].clone().requires_grad_(True)
        v = fn(p)
        v.backward()
        assert torch.allclose(v, fix[name]["value"], rtol=1e-6), name
        assert rel_err(p.grad, fix[name]["grad"]) <= 1e-6, name
    m = O.nds_mask(fix["spec"] - fix["ysp"])
    assert torch.equal(m, fix["mask_special"])
    assert np.array_equal(O.nds_mask_numpy(fix["spec"].numpy(), fix["ysp"].numpy()), fix["mask_special"].numpy())
    assert m.view(-1)[:6].tolist() == [False, False, True, True, False, True]


def test_irfft2_contract_numpy_matches_torch():
    g = torch.Generator().manual_seed(3)
    re, im = torch.randn(2, 3, 16, 9, generator=g), torch.randn(2, 3, 16, 9, generator=g)
    want = torch.fft.irfft2(torch.complex(re, im), s=(16, 16), dim=(2, 3), norm="ortho")
    got = O.irfft2_contract_numpy(re.numpy(), im.numpy(), 16, 16)
    assert np.abs(got - want.numpy()).max() <= 1e-5


def test_oracle_vs_reference_outputs(seeded_sd):
    """The oracle's d_loss / g_loss equal, bit for bit, what the live reference computed on the same weights, inputs and
    dropout masks.  The reference's Ablation_CLS_SEG_REC_NDS_RC_ResFFT builds MTD_GAN_Method's generator and
    discriminator in the same order and sums the same loss terms, so its row of ablation.pt (make_golden_ablation.py)
    holds the reference's initial state and its d_loss / g_loss totals and terms."""
    fix = load("ablation.pt")["Ablation_CLS_SEG_REC_NDS_RC_ResFFT"]
    assert list(seeded_sd.keys()) == list(fix["state"].keys())
    for k, v in seeded_sd.items():
        check_summary(v, fix["state"][k], 0.0, k)                  # drop-in init == reference init, bit for bit
    x, y = O.synthetic_pair(2, 64, seed=77)
    masks = [drop_mask(2, 900 + i) for i in range(5)]             # the reference's dropout masks, in call order
    sd = {k: v.clone() for k, v in seeded_sd.items()}
    l_or, d_or = O.d_loss(sd, x, y, True, masks[:4])
    assert float(l_or[0] + l_or[1] + l_or[2]) == fix["d_total"]
    assert list(d_or.keys()) == list(fix["d_details"].keys())
    for k, v in fix["d_details"].items():
        assert float(d_or[k]) == v, k
    g_or, gd_or = O.g_loss(sd, x, y, True, masks[4])
    assert float(g_or) == fix["g_total"]
    assert list(gd_or.keys()) == list(fix["g_details"].keys())
    for k, v in fix["g_details"].items():
        assert float(gd_or[k]) == v, k
