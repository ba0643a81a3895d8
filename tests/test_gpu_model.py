"""GPU parity tests of the drop-in modules (generator, discriminator, method wrapper, PCGrad, one full
training step) against the golden vectors generated from the live reference and against the CPU oracle on
the same seeded inputs.  Tolerances are the north_star's: fp32 path <= 1e-4 (norm-wise relative error),
stated per check; bit-exact for the NDS mask (test_gpu_kernels.py)."""
import random

import pytest
import torch

from _golden_util import GradTally, check_summary, load, rel_err
from oracle import mtdgan_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def drop_mask(b, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, 512, generator=g) >= 0.3).float() / 0.7


def seeded_model():
    from arch.Ours.networks import MTD_GAN_Method
    torch.manual_seed(2024)
    random.seed(2024)
    return MTD_GAN_Method().to(DEV)


class Tol:
    """Per-mode tolerances (norm-wise relative errors).
    simt: exact fp32 SIMT kernels everywhere — the north_star's 1e-4 on outputs / losses / gradients.
    tc3 : tcgen05 error-compensated 3xTF32 on the contraction layers (the default): fp32-grade outputs (3e-4);
          gradients within the north_star's tensor-core bound 2e-3 (a 1e-5 perturbation flips more ReLU masks than
          fp32's 1e-7, and single flips move small-norm gradient sums by ~1e-3).
    tc1 : plain TF32 opt-in fast mode: outputs 5e-3 after 20-64 layers; gradients of a deep ReLU net move by several
          per cent under ANY plain-TF32 evaluation (cuDNN's included), so only a sanity bound (1e-1, median 1e-2)."""
    def __init__(self, mode):
        self.mode = mode
        self.out = {"simt": 1e-4, "tc3": 3e-4, "tc1": 1e-2}[mode]
        # BASELINE configs[1] (1x512x512 generator forward): north_star's 1e-4 in both fp32-grade modes
        self.out512 = {"simt": 1e-4, "tc3": 1e-4, "tc1": 1e-2}[mode]
        # per-tensor bound; the MEDIAN over tensors (below) is the sharp check (measured ~3e-7 in simt mode).  With 4
        # samples a deep discriminator layer sees 4-16 pixels, so one flipped LeakyReLU decision (forward sums differ in
        # the last bit between runs: fp32 atomics) moves a tensor by a few 1e-4 -- hence 1e-3, not 2e-4, per tensor.
        self.grad = {"simt": 1e-3, "tc3": 2e-3, "tc1": 1e-1}[mode]
        self.median = {"simt": 1e-4, "tc3": 1e-3, "tc1": 1e-2}[mode]   # tc3: weight gradients run in plain TF32 (2e-3 class)


@pytest.fixture(params=["simt", "tc3", "tc1"])
def conv_mode(request):
    from mtdgan_b200 import ops
    if request.param == "simt":
        ops.set_conv_mode("simt")
    else:
        ops.set_conv_mode("auto", 3 if request.param == "tc3" else 1)
    yield Tol(request.param)
    ops.set_conv_mode("auto", 3)


@pytest.fixture()
def masks():
    from mtdgan_b200 import networks as NW
    queue = []
    NW.set_dropout_mask_provider(lambda b, n, dev: queue.pop(0).to(dev) if queue else None)
    yield queue
    NW.set_dropout_mask_provider(None)


def test_generator_forward_64(conv_mode):
    m = seeded_model().eval()
    x = O.synthetic_pair(2, 64, seed=11)[0].to(DEV)
    with torch.no_grad():
        out = m.Generator(x)
    assert out.shape == (2, 1, 64, 64) and float(out.min()) >= 0.0
    assert rel_err(out, load("gen_fwd_64.pt")["out"]) <= conv_mode.out


def test_generator_forward_512(conv_mode):
    m = seeded_model().eval()
    x = O.synthetic_pair(1, 512, seed=12)[0].to(DEV)
    with torch.no_grad():
        out = m.Generator(x)
    err = rel_err(out, load("gen_fwd_512.pt")["out"])          # fp32 fixture from the live reference
    print("generator 512x512 forward (%s): rel err %.2e" % (conv_mode.mode, err))
    assert err <= conv_mode.out512
    # batch independence: slices of a batch equal single-slice calls (inference shards by slice)
    with torch.no_grad():
        xb = torch.cat([x, x.flip(-1)], 0)
        ob = m.Generator(xb)
    assert rel_err(ob[:1], out) <= 1e-5


@pytest.mark.parametrize("B,S", [(2, 64), (1, 128)], ids=["2x64", "1x128"])     # training patches: 64^2, 128^2
def test_generator_backward_vs_oracle(B, S, conv_mode):
    if conv_mode.mode == "tc1":
        pytest.skip("plain-TF32 opt-in mode: gradients of a 64-layer ReLU net are only sanity-checked at kernel level")
    m = seeded_model()
    x = O.synthetic_pair(B, S, seed=41)[0]
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in m.Generator.state_dict().items()}
    g = torch.Generator().manual_seed(42)
    w = torch.randn(B, 1, S, S, generator=g)
    (O.generator_forward(sd, x) * w).sum().backward()
    out = m.Generator(x.to(DEV))
    (out * w.to(DEV)).sum().backward()
    # noise floor: the oracle's own fp32-vs-fp64 gap on the same weights (ReLU-mask flips, see _golden_util)
    sd64 = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
    (O.generator_forward(sd64, x.double()) * w.double()).sum().backward()
    tally = GradTally()
    floors = []
    for k, p in m.Generator.named_parameters():
        floor = rel_err(sd[k].grad, sd64[k].grad)
        floors.append(floor)
        tally.add(k, rel_err(p.grad, sd[k].grad), max(conv_mode.grad, 30 * floor))
    # where the oracle's own fp32 evaluation misses the mode's median bound (1x128: median fp32-vs-fp64 gap 1.7e-4, more
    # ReLU units to flip), the bound is twice that gap: the GPU is compared with the fp32 evaluation, two draws of it
    ref_median = sorted(floors)[len(floors) // 2]
    print("oracle fp32-vs-fp64 median gap %.2e" % ref_median)
    tally.finish(conv_mode.median if ref_median <= conv_mode.median else 2 * ref_median)


def test_discriminator_vs_golden(masks, conv_mode):
    fix = load("disc_64.pt")
    m = seeded_model()
    D = m.Discriminator.train()
    y = O.synthetic_pair(2, 64, seed=13)[1].to(DEV)
    masks.append(drop_mask(2, 14))
    enc, dec, rec = D(y)
    assert enc.shape == (2, 1) and dec.shape == (2, 1, 64, 64) and rec.shape == (2, 1, 64, 64)
    for got, key in ((enc, "enc"), (dec, "dec"), (rec, "rec")):
        assert rel_err(got, fix[key]) <= conv_mode.out, key
    g = torch.Generator().manual_seed(15)
    a, b, c = (torch.randn(s, generator=g).to(DEV) for s in (enc.shape, dec.shape, rec.shape))
    ((enc * a).sum() + (dec * b).sum() / 64 + (rec * c).sum() / 64).backward()
    tally = GradTally()
    for k, p in D.named_parameters():
        if k in fix["grads"]:
            if conv_mode.mode != "tc1":
                check_summary(p.grad, fix["grads"][k], conv_mode.grad, k, tally=tally)
        else:
            assert p.grad is None, k
    if conv_mode.mode != "tc1":
        tally.finish()
    for k, v in D.named_buffers():
        check_summary(v, fix["buffers"][k], 1e-5, k)
    D.eval()
    with torch.no_grad():
        e2, d2, r2 = D(y)
    tol = conv_mode.out
    assert rel_err(e2, fix["eval_enc"]) <= tol and rel_err(d2, fix["eval_dec"]) <= tol and rel_err(r2, fix["eval_rec"]) <= tol
    with pytest.raises(RuntimeError):
        D(torch.zeros(1, 1, 512, 512, device=DEV))            # D only accepts 64 x 64 (SURVEY §3.4)


def test_full_train_step_b4_vs_golden(masks, conv_mode):
    if conv_mode.mode == "tc1":
        pytest.skip("plain-TF32 opt-in mode is not a parity mode for training (see Tol)")
    """BASELINE configs[0]: one MTD_GAN_Method train step (engine.py:40-55) on 4 synthetic 64^2 patches."""
    from module.weight_methods import WeightMethods
    fix = load("train_step_b4.pt")
    m = seeded_model().train()
    D, G = m.Discriminator, m.Generator
    x, y = (t.to(DEV) for t in O.synthetic_pair(4, 64, seed=1234))
    masks.extend(drop_mask(4, 21 + i) for i in range(5))
    opt_D = torch.optim.AdamW(D.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4)
    opt_G = torch.optim.AdamW(G.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4)
    wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
    random.seed(99)
    opt_D.zero_grad(); D.zero_grad()
    d_losses, det = m.d_loss(x, y)
    assert d_losses.shape == (3,)
    cm = conv_mode
    assert torch.allclose(d_losses.cpu()[:2], fix["d_losses"][:2], rtol=cm.out, atol=1e-10)
    for k, v in fix["d_details"].items():
        # terms that are squares of ~1e-6 quantities (consistency, fake_enc at init) carry twice the relative error
        # of the tiny outputs they are built from
        assert torch.allclose(det[k].cpu(), v, rtol=(10 if float(v) > 1e-3 else 300) * cm.out, atol=1e-10), k
    loss_D, extra = wm.backward(losses=d_losses, shared_parameters=list(D.shared_parameters()),
                                task_specific_parameters=list(D.task_specific_parameters()),
                                last_shared_parameters=list(D.last_shared_parameters()))
    assert loss_D is None and extra == {}
    tally = GradTally()
    for k, p in D.named_parameters():
        if fix["d_grads"][k] is None:
            assert p.grad is None, k                               # c_fc.* (SURVEY Q1)
        else:
            check_summary(p.grad, fix["d_grads"][k], cm.grad, k, noise=fix["d_grads_noise"][k], tally=tally)
    tally.finish()
    opt_D.step()
    opt_G.zero_grad(); G.zero_grad()
    g_loss, gdet = m.g_loss(x, y)
    assert abs(float(g_loss) - float(fix["g_loss"])) <= cm.out * abs(float(fix["g_loss"]))
    for k, v in fix["g_details"].items():
        assert torch.allclose(gdet[k].cpu(), v, rtol=cm.out, atol=1e-8), k
    g_loss.backward()
    tally = GradTally()
    errs = [check_summary(p.grad, fix["g_grads"][k], cm.grad, k, noise=fix["g_grads_noise"][k], tally=tally)[0]
            for k, p in G.named_parameters()]
    tally.finish()
    assert sorted(errs)[len(errs) // 2] <= cm.median     # median norm error over the 128 generator tensors
    opt_G.step()
    sd = m.state_dict()
    # AdamW's first step moves every entry by ~lr*sign(g) whatever |g| is, so a near-zero gradient entry whose sign
    # differs moves that entry by 2*lr: weights of RMS ~1e-2 stay within 2e-3, but zero-initialised biases (every entry
    # is +-lr after the step) are only comparable as a population -- judged like the gradients (GradTally)
    tally = GradTally(frac_outliers=0.04, gross=0.5, gross_spectral_bias=0.5)
    for k, s in fix["state_after"].items():
        if k.endswith("bias"):
            check_summary(sd[k], s, 2e-3 if cm.mode != "tc1" else 4e-2, k, tally=tally)
        else:
            check_summary(sd[k], s, 2e-3 if cm.mode != "tc1" else 4e-2, k)
    tally.finish()


def test_two_steps_fused_adamw_runs_and_decreases_nothing_nan():
    """Two steps with the fused optimizer: finite losses, weights move, u/v buffers stay unit-norm."""
    from module.weight_methods import WeightMethods
    from mtdgan_b200.optim import FusedAdamW
    m = seeded_model().train()
    D, G = m.Discriminator, m.Generator
    x, y = (t.to(DEV) for t in O.synthetic_pair(4, 64, seed=5))
    opt_D = FusedAdamW([{"params": D.parameters()}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
    opt_G = FusedAdamW(G.parameters(), lr=1e-4, weight_decay=5e-4)
    wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
    w0 = D.conv12.weight_orig.detach().clone()
    for _ in range(2):
        opt_D.zero_grad(); D.zero_grad()
        d_losses, _ = m.d_loss(x, y)
        wm.backward(losses=d_losses, shared_parameters=list(D.shared_parameters()),
                    task_specific_parameters=list(D.task_specific_parameters()),
                    last_shared_parameters=list(D.last_shared_parameters()))
        opt_D.step()
        opt_G.zero_grad(); G.zero_grad()
        g_loss, _ = m.g_loss(x, y)
        g_loss.backward()
        opt_G.step()
        assert torch.isfinite(d_losses).all() and torch.isfinite(g_loss)
    assert not torch.equal(w0, D.conv12.weight_orig)
    assert abs(float(D.conv12.weight_u.norm()) - 1.0) < 1e-4
    assert D.c_fc.weight_orig.grad is None


def test_cuda_graph_step_matches_eager():
    """GraphedTrainStep: capture + replay of the whole train step reproduces eager execution (dropout disabled so
    both consume no torch RNG; PCGrad orders re-seeded before the compared steps).  The capture restores weights,
    optimizer state and RNGs, so replay k == eager step k: two consecutive steps are compared."""
    from module.weight_methods import WeightMethods
    from mtdgan_b200.graphs import GraphedTrainStep
    from mtdgan_b200.optim import FusedAdamW
    x, y = (t.to(DEV) for t in O.synthetic_pair(4, 64, seed=9))
    results = []
    for use_graph in (False, True):
        m = seeded_model().train()
        m.Discriminator.c_drop.p = 0.0
        D, G = m.Discriminator, m.Generator
        opt_D = FusedAdamW([{"params": list(D.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
        opt_G = FusedAdamW(G.parameters(), lr=1e-4, weight_decay=5e-4)
        wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
        runner = GraphedTrainStep(m, opt_D, opt_G, wm)
        if use_graph:
            runner.capture(x, y, warmup=2)          # two eager warm-up steps + the capture pass, state restored afterwards
        random.seed(1)
        runner(x, y)
        random.seed(2)
        dl, _, gl, _ = runner(x, y)                 # second step: replay vs eager
        torch.cuda.synchronize()
        results.append((dl.clone().cpu(), gl.clone().cpu(), {k: v.detach().clone().cpu() for k, v in m.state_dict().items()}))
    (dl_e, gl_e, sd_e), (dl_g, gl_g, sd_g) = results
    assert torch.allclose(dl_e[:2], dl_g[:2], rtol=1e-4, atol=1e-10) and torch.allclose(gl_e, gl_g, rtol=1e-4)
    # AdamW's first steps move every entry by ~ +-lr whatever the gradient magnitude, so a sign flip of a ~0 gradient
    # entry (fp32 atomics order differs between runs) shows up as 2*lr on zero-initialised biases: bound the bulk, not
    # the worst element
    errs = sorted(rel_err(sd_g[k], sd_e[k]) for k in sd_e)
    assert errs[len(errs) // 2] <= 1e-4 and errs[int(len(errs) * 0.9)] <= 5e-2, (errs[len(errs) // 2], errs[-1])
    worst_abs = max(float((sd_g[k].double() - sd_e[k].double()).abs().max()) for k in sd_e if not k.endswith(("weight_u", "weight_v")))
    assert worst_abs <= 2 * 2 * 1e-4 + 1e-6, worst_abs          # <= 2*lr per step per element


@pytest.mark.parametrize("mode", ["simt", "tc3"])
def test_discriminator_grouped_pass_equals_separate_calls(masks, mode):
    """D(cat[a, b], groups=2) == (D(a), D(b)) called one after the other: outputs, spectral-norm buffers and the
    parameter gradients of a loss over both (d_loss batches the reference's call pairs this way).  In exact-fp32 mode
    the two evaluations differ only by summation order; in the default tensor-core mode the weight gradients are
    plain TF32 (2e-3 class) and the GEMMs are tiled differently (3 vs 6 samples per launch)."""
    import copy
    from mtdgan_b200 import ops
    ops.set_conv_mode("simt" if mode == "simt" else "auto", 3)
    try:
        m1 = seeded_model().train()
        D1 = m1.Discriminator
        D2 = copy.deepcopy(D1)
        a, b = (t.to(DEV) for t in O.synthetic_pair(3, 64, seed=77))
        mk = [drop_mask(3, 31), drop_mask(3, 32)]
        masks.extend([mk[0], mk[1]])
        e1, d1, r1 = D1(a)
        e2, d2, r2 = D1(b)
        masks.extend([mk[0], mk[1]])
        e, d, r = D2(torch.cat([a, b], 0), groups=2)
        for got, ref in ((e, torch.cat([e1, e2])), (d, torch.cat([d1, d2])), (r, torch.cat([r1, r2]))):
            assert rel_err(got, ref) <= 1e-4          # x_enc is ~1e-6 at initialisation: fp32 noise of the last layer
        for (k, v1), (_, v2) in zip(D1.named_buffers(), D2.named_buffers()):
            assert rel_err(v2, v1) <= 1e-6, k
        g = torch.Generator().manual_seed(3)
        we, wd, wr = (torch.randn(s, generator=g).to(DEV) for s in (e.shape, d.shape, r.shape))
        ((torch.cat([e1, e2]) * we).sum() + (torch.cat([d1, d2]) * wd).sum() / 64 + (torch.cat([r1, r2]) * wr).sum() / 64).backward()
        ((e * we).sum() + (d * wd).sum() / 64 + (r * wr).sum() / 64).backward()
        tally = GradTally()
        for (k, p1), (_, p2) in zip(D1.named_parameters(), D2.named_parameters()):
            if p1.grad is None:
                assert p2.grad is None, k
            else:
                tally.add(k, rel_err(p2.grad, p1.grad), 2e-2)
        # Forward values differ in the last fp32 bits between the two evaluations, so individual LeakyReLU decisions flip:
        # per-tensor agreement is statistical (GradTally); a wrong per-group sigma / u / v would shift EVERY
        # spectrally-normalised weight gradient by O(1).
        errs = tally.finish(1e-4 if mode == "simt" else 5e-3)
        print("grouped-vs-separate gradient errors (%s): median %.2e, p90 %.2e, max %.2e"
              % (mode, errs[len(errs) // 2], errs[int(len(errs) * 0.9)], errs[-1]))
    finally:
        ops.set_conv_mode("auto", 3)


def _fixed_masks(b, n=5, seed0=500):
    return [drop_mask(b, seed0 + i) for i in range(n)]


def oracle_d_grads(sd0, x, y, mk, seed, dtype):
    """d_losses and the discriminator gradients the reference's `weight_method.backward` leaves in `.grad`
    (post-PCGrad on the shared set, sum-loss gradients on the task-specific set; weight_methods.py:429-447)."""
    sd = {k: (v.to(dtype) if v.is_floating_point() else v.clone()) for k, v in sd0.items()}
    for k, v in sd.items():
        if not k.endswith(("weight_u", "weight_v")):
            v.requires_grad_(True)
    dn = "Discriminator."
    shared = [sd[dn + n] for n in O.d_shared_names()]
    ts = [sd[dn + n] for n in O.d_task_specific_names()]
    random.seed(seed)
    dl, _ = O.d_loss(sd, x.to(dtype), y.to(dtype), True, [t.to(dtype) for t in mk[:4]])
    grads = [torch.autograd.grad(l, shared, retain_graph=True) for l in dl]
    merged = O.pcgrad_project_lists(grads, "sum")
    tsg = torch.autograd.grad(dl.sum(), ts)
    out = {n: g for n, g in zip(O.d_shared_names(), merged)}
    out.update({n: g for n, g in zip(O.d_task_specific_names(), tsg)})
    return dl.detach(), out


def test_graph_replayed_b20_step_vs_oracle():
    """The BENCHMARKED configuration (BASELINE configs[2]): 20 patches, whole step replayed as one CUDA graph with
    grouped discriminator passes, generator-forward reuse, side-stream weight gradients and fused AdamW -- compared
    with the CPU oracle's train step (engine.py:40-55 restated) on the same inputs, weights, dropout masks and PCGrad
    visit orders: d_losses, all 14 details, post-PCGrad / task-specific / generator gradients, weights after the step."""
    from module.weight_methods import WeightMethods
    from mtdgan_b200 import networks as NW
    from mtdgan_b200.graphs import GraphedTrainStep
    from mtdgan_b200.optim import FusedAdamW
    from oracle.train_step import OracleTrainer
    B = 20
    x, y = O.synthetic_pair(B, 64, seed=1234)
    m = seeded_model().train()
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    D, G = m.Discriminator, m.Generator
    opt_D = FusedAdamW([{"params": list(D.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
    opt_G = FusedAdamW(G.parameters(), lr=1e-4, weight_decay=5e-4)
    wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
    mk = _fixed_masks(B)
    mk_dev = [t.to(DEV) for t in mk]
    calls = [0]

    def provider(b, n, dev):                 # d_loss: D(real), D(fake), D(clip real_rec), D(clip fake_rec); g_loss: D(fake)
        t = mk_dev[calls[0] % 5]
        calls[0] += 1
        return t

    NW.set_dropout_mask_provider(provider)
    try:
        runner = GraphedTrainStep(m, opt_D, opt_G, wm)
        runner.capture(x.to(DEV), y.to(DEV), warmup=2)          # state is restored: the first replay is step 1
        for k, v in m.state_dict().items():
            assert torch.equal(v.cpu(), sd0[k]), f"capture disturbed {k}"
        random.seed(4242)
        dl, ddet, gl, gdet = runner(x.to(DEV), y.to(DEV))
        torch.cuda.synchronize()
    finally:
        NW.set_dropout_mask_provider(None)
    got = {"dl": dl.cpu().clone(), "gl": gl.cpu().clone(), "ddet": {k: v.detach().cpu().clone() for k, v in ddet.items()},
           "gdet": {k: v.detach().cpu().clone() for k, v in gdet.items()},
           "dgrad": {k: p.grad.detach().cpu().clone() for k, p in D.named_parameters() if p.grad is not None},
           "ggrad": {k: p.grad.detach().cpu().clone() for k, p in G.named_parameters() if p.grad is not None},
           "sd": {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}}

    # ---- oracle, fp32 and (noise floor) fp64, same masks / orders
    def oracle_run(dtype):
        tr = OracleTrainer({k: v.to(dtype) if v.is_floating_point() else v for k, v in sd0.items()})
        random.seed(4242)
        dl_, dd_, gl_, gd_ = tr.step(x.to(dtype), y.to(dtype), dropout_masks=[t.to(dtype) for t in mk])
        return tr, dl_, dd_, gl_, gd_

    tr32, dl32, dd32, gl32, gd32 = oracle_run(torch.float32)
    tol = Tol("tc3")
    print("B=20 replay d_losses", got["dl"].tolist(), "oracle", dl32.tolist(), "g_loss", float(got["gl"]), float(gl32))
    assert torch.allclose(got["dl"][:2], dl32[:2], rtol=tol.out, atol=1e-10)
    for k, v in dd32.items():
        assert torch.allclose(got["ddet"][k], v.detach(), rtol=(10 if float(v) > 1e-3 else 300) * tol.out, atol=1e-10), k
    assert abs(float(got["gl"]) - float(gl32)) <= tol.out * abs(float(gl32))
    for k, v in gd32.items():
        assert torch.allclose(got["gdet"][k], v.detach(), rtol=tol.out, atol=1e-8), k
    # generator gradients: still on the oracle's leaves after its step
    tr64, *_ = oracle_run(torch.float64)
    tally = GradTally()
    for k, g in got["ggrad"].items():
        g32, g64 = tr32.sd["Generator." + k].grad, tr64.sd["Generator." + k].grad
        tally.add("G." + k, rel_err(g, g32), max(tol.grad, 30 * rel_err(g32, g64)))
    tally.finish(tol.median)
    # discriminator gradients left by the replayed step (g_loss does not touch them: its D pass runs with frozen weights)
    _, d32 = oracle_d_grads(sd0, x, y, mk, 4242, torch.float32)
    _, d64 = oracle_d_grads(sd0, x, y, mk, 4242, torch.float64)
    tally = GradTally()
    for k, g in got["dgrad"].items():
        tally.add("D." + k, rel_err(g, d32[k]), max(tol.grad, 30 * rel_err(d32[k], d64[k])))
    assert set(got["dgrad"]) == set(d32), set(got["dgrad"]) ^ set(d32)
    tally.finish(tol.median)
    # weights after the full step (D and G): AdamW's first step moves every entry by ~lr whatever |g| is, so compare
    # as a population (a sign flip of a ~0 gradient entry is 2*lr on that entry)
    errs, worst_abs = [], 0.0
    for k, v in got["sd"].items():
        if k.endswith(("weight_u", "weight_v")):
            assert rel_err(v, tr32.sd[k]) <= 1e-3, k
            continue
        errs.append(rel_err(v, tr32.sd[k].detach()))
        worst_abs = max(worst_abs, float((v.double() - tr32.sd[k].detach().double()).abs().max()))
    errs.sort()
    print("weights after step: median rel err %.2e, p90 %.2e, worst abs %.2e" % (errs[len(errs) // 2], errs[int(len(errs) * 0.9)], worst_abs))
    assert errs[len(errs) // 2] <= 1e-4 and worst_abs <= 2 * 1e-4 + 1e-6


def test_b20_post_pcgrad_gradients_vs_oracle(masks):
    """Post-PCGrad shared gradients and task-specific gradients of the discriminator at the benchmarked batch (20),
    eager launches of the same kernels the graph replays, against the oracle with its fp32-vs-fp64 gap as noise floor."""
    from module.weight_methods import WeightMethods
    B = 20
    x, y = O.synthetic_pair(B, 64, seed=1234)
    m = seeded_model().train()
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    D = m.Discriminator
    mk = _fixed_masks(B, 4, 700)
    masks.extend(t.clone() for t in mk)
    wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
    random.seed(99)
    d_losses, _ = m.d_loss(x.to(DEV), y.to(DEV))
    wm.backward(losses=d_losses, shared_parameters=list(D.shared_parameters()),
                task_specific_parameters=list(D.task_specific_parameters()), last_shared_parameters=list(D.last_shared_parameters()))

    dl32, g32 = oracle_d_grads(sd0, x, y, mk, 99, torch.float32)
    _, g64 = oracle_d_grads(sd0, x, y, mk, 99, torch.float64)
    tol = Tol("tc3")
    assert torch.allclose(d_losses.detach().cpu()[:2], dl32[:2], rtol=tol.out, atol=1e-10)
    tally = GradTally()
    for k, p in D.named_parameters():
        if k in g32:
            tally.add(k, rel_err(p.grad, g32[k]), max(tol.grad, 30 * rel_err(g32[k], g64[k])))
        else:
            assert p.grad is None, k
    tally.finish(tol.median)


def test_batched_inference_512_vs_oracle(conv_mode):
    """BASELINE configs[4] path: a batch of 512x512 slices through the CUDA-graph inference runner (micro-batches, zero
    padded tail) equals the oracle's generator forward slice by slice, <= 1e-4 in the fp32-grade modes."""
    from mtdgan_b200.inference import GraphedGenerator
    m = seeded_model().eval()
    n = 8 if conv_mode.mode == "tc3" else 3
    x = O.synthetic_pair(n, 512, seed=31)[0]
    sd = {k: v.detach().cpu() for k, v in m.Generator.state_dict().items()}
    with torch.no_grad():
        want = torch.cat([O.generator_forward(sd, x[i:i + 1]) for i in range(n)])
    runner = GraphedGenerator(m.Generator, 512, 512, micro_batch=3).capture()
    got = runner(x.to(DEV))
    torch.cuda.synchronize()
    errs = [rel_err(got[i], want[i]) for i in range(n)]
    print("batched 512x512 inference (%s): per-slice rel err max %.2e" % (conv_mode.mode, max(errs)))
    assert max(errs) <= conv_mode.out512
    got2 = runner(x.to(DEV))                       # replays are idempotent
    assert torch.equal(got, got2)


def test_captured_step_follows_lr_schedule():
    """ADVICE r1: the learning rate must not be frozen into the captured graph.  Capture at lr 1e-4, then set 3e-5 (what
    scheduler_D / scheduler_G do every epoch) and replay: weights must equal an eager run with the same schedule."""
    from module.weight_methods import WeightMethods
    from mtdgan_b200.graphs import GraphedTrainStep
    from mtdgan_b200.optim import FusedAdamW
    x, y = (t.to(DEV) for t in O.synthetic_pair(4, 64, seed=9))
    res = []
    for use_graph in (False, True):
        m = seeded_model().train()
        m.Discriminator.c_drop.p = 0.0
        D, G = m.Discriminator, m.Generator
        opt_D = FusedAdamW([{"params": list(D.parameters())}, {"params": [], "lr": 0.025}], lr=1e-4, weight_decay=5e-4)
        opt_G = FusedAdamW(G.parameters(), lr=1e-4, weight_decay=5e-4)
        wm = WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))
        runner = GraphedTrainStep(m, opt_D, opt_G, wm)
        if use_graph:
            runner.capture(x, y, warmup=1)
        for o in (opt_D, opt_G):
            o.param_groups[0]["lr"] = 3e-5
        w0 = {k: v.detach().clone() for k, v in m.state_dict().items()}
        random.seed(3)
        runner(x, y)
        torch.cuda.synchronize()
        # AdamW's first step moves each entry by ~lr * sign(g): the mean absolute update measures the lr in effect
        moved = torch.cat([(v - w0[k]).abs().flatten() for k, v in m.state_dict().items()
                           if k.endswith(("weight_orig", "weight")) and v.dim() == 4])
        res.append(float(moved.mean()))
        big = [(k, float((v - w0[k]).abs().max())) for k, v in m.state_dict().items()
               if not k.endswith(("weight_u", "weight_v")) and float((v - w0[k]).abs().max()) > 2.5 * 3e-5]
        print("graph" if use_graph else "eager", "parameters that moved by more than 2.5 x lr:", len(big), big[:8])
    print("mean |dw| after one step at lr 3e-5: eager %.3e, graph %.3e" % tuple(res))
    assert abs(res[1] - res[0]) <= 0.05 * res[0] and res[0] < 5e-5
