"""PCGrad's task-specific gradients folded from the per-task backward passes (ops.fold_task_grads): the activation
backward with a fold output against a torch restatement, the launch count of the driver's backward against the three
per-task passes alone, and the folded gradients against the oracle's autograd.grad(losses.sum(), task_specific)."""
import random

import pytest
import torch

from _golden_util import rel_err
from oracle import mtdgan_oracle as O
from test_gpu_model import _fixed_masks, oracle_d_grads, seeded_model

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("act", [0, 2])
@pytest.mark.parametrize("acc_first", [0, 1])
@pytest.mark.parametrize("groups", [1, 2])
@pytest.mark.parametrize("M,N", [(2 * 3 * 32 * 32, 64), (2 * 5 * 16 * 16, 1)])
def test_act_bwd_acc_matches_reference(M, N, groups, acc_first, act):
    """mtd_act_bwd_acc: dz as mtd_act_bwd writes it, acc (+)= dz / sigma_g, bias gradient and <G, W~> coefficients
    accumulated onto what is already there."""
    from mtdgan_b200._ext import call, fptr, stream
    g = torch.Generator().manual_seed(M + N + 7 * groups + act)
    ypre = torch.randn(M, N, generator=g, dtype=torch.float64).float()
    bias = (torch.randn(N, generator=g, dtype=torch.float64) * 0.1).float()
    dy = torch.randn(M, N, generator=g, dtype=torch.float64).float()
    acc0 = torch.randn(M, N, generator=g, dtype=torch.float64).float()
    db0 = torch.randn(N, generator=g, dtype=torch.float64).float()
    zw0 = torch.randn(groups, generator=g, dtype=torch.float64)
    sc = torch.tensor([0.5 + 0.25 * k for k in range(groups)])
    y = torch.where(ypre > 0, ypre, 0.2 * ypre) if act == 2 else ypre
    dz_ref = dy * torch.where(y > 0, 1.0, 0.2).float() if act == 2 else dy             # fp32, as the kernel computes it
    rowscale = sc.repeat_interleave(M // groups).reshape(M, 1).double()
    acc_ref = dz_ref.double() * rowscale + (0 if acc_first else acc0.double())
    db_ref = db0.double() + dz_ref.double().sum(0)
    terms = (dz_ref.double() * (ypre.double() - bias.double())).reshape(groups, -1)
    zw_ref = zw0 + terms.sum(1)

    dyc, yc, bc, scc = dy.to(DEV), y.to(DEV), bias.to(DEV), sc.to(DEV)
    dz = torch.full_like(dyc, float("nan"))
    acc = acc0.to(DEV) if not acc_first else torch.full_like(dyc, float("nan"))
    db, zw = db0.to(DEV), zw0.to(DEV)
    call("mtd_act_bwd_acc", fptr(dyc), fptr(yc), fptr(dz) if act else None, fptr(acc), acc_first, fptr(db), fptr(bc),
         zw.data_ptr(), fptr(scc), groups, M, N, act, 0.2, stream())
    torch.cuda.synchronize()
    if act:
        assert torch.equal(dz.cpu(), dz_ref)
    assert rel_err(acc, acc_ref) <= 1e-6
    # column sums in fp32 (atomics, any order): bound by the cancellation-free magnitude, like zw
    assert float((db.cpu() - db_ref).abs().max()) <= 1e-6 * float(db0.abs().max() + dz_ref.abs().sum(0).max())
    # y_pre is recovered from y (LeakyReLU inverted) and each term is an fp32 product: bound by the cancellation-free sum
    assert float((zw.cpu() - zw_ref).abs().max()) <= 1e-6 * float(terms.abs().sum(1).max())

    # layer without spectral norm and without activation (heads, UpsampleBlock 1x1): acc (+)= dy, no y, no zw
    acc2 = acc0.to(DEV) if not acc_first else torch.full_like(dyc, float("nan"))
    db2 = db0.to(DEV)
    call("mtd_act_bwd_acc", fptr(dyc), None, None, fptr(acc2), acc_first, fptr(db2), None, None, None, groups, M, N, 0, 0.2,
         stream())
    torch.cuda.synchronize()
    assert torch.equal(acc2.cpu(), dy + (0 if acc_first else acc0))
    db2_ref = db0.double() + dy.double().sum(0)
    assert float((db2.cpu() - db2_ref).abs().max()) <= 1e-6 * float(db0.abs().max() + dy.abs().sum(0).max())


def _d_setup(B):
    from module.weight_methods import WeightMethods
    m = seeded_model().train()
    x, y = O.synthetic_pair(B, 64, seed=1234)
    return m, x.to(DEV), y.to(DEV), WeightMethods('pcgrad', n_tasks=3, device=torch.device(DEV))


_COUNTED = ("mtd_conv_dgrad", "mtd_act_bwd", "mtd_upsample2x_bwd")


def _count(trace):
    n = sum(1 for name, _ in trace if name.startswith(_COUNTED))
    return n + sum(1 for name, args in trace if name == "mtd_pixel_shuffle2" and args[-2] == 1)     # backward direction


def test_fold_runs_no_extra_backward_pass():
    """The driver's backward issues exactly the data-gradient, activation-backward and resampling-backward launches of
    the three per-task passes over the shared parameters: nothing is re-walked for the task-specific gradients."""
    from mtdgan_b200 import _ext
    from mtdgan_b200.ops import deferred_wgrad_finish, wgrad_only_for
    B = 4
    m, x, y, wm = _d_setup(B)
    D = m.Discriminator
    shared, ts = list(D.shared_parameters()), list(D.task_specific_parameters())
    torch.manual_seed(3)
    random.seed(3)
    d_losses, _ = m.d_loss(x, y)
    _ext.start_trace()
    wm.backward(losses=d_losses, shared_parameters=shared, task_specific_parameters=ts)
    got = _count(_ext.stop_trace())
    assert all(p.grad is not None for p in ts)

    m2, _, _, _ = _d_setup(B)
    shared2 = list(m2.Discriminator.shared_parameters())
    torch.manual_seed(3)
    d_losses2, _ = m2.d_loss(x, y)
    _ext.start_trace()
    with wgrad_only_for(shared2):
        for l in d_losses2:
            with deferred_wgrad_finish():
                torch.autograd.grad(l, shared2, retain_graph=True)
    want = _count(_ext.stop_trace())
    torch.cuda.synchronize()
    assert got == want, (got, want)


def test_simt_task_specific_grads_vs_oracle():
    """Exact-fp32 kernels: the folded task-specific gradients equal the oracle's autograd.grad(losses.sum(), ts) to
    fp32 summation order, so a wrong 1/sigma, <G, W~> coefficient or bias term shows up as an O(1) error."""
    from mtdgan_b200 import networks as NW, ops
    B = 4
    mk = _fixed_masks(B, 4, 800)
    queue = [t.clone() for t in mk]
    NW.set_dropout_mask_provider(lambda b, n, dev: queue.pop(0).to(dev) if queue else None)
    ops.set_conv_mode("simt")
    try:
        m, x, y, wm = _d_setup(B)
        sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
        D = m.Discriminator
        random.seed(17)
        d_losses, _ = m.d_loss(x, y)
        wm.backward(losses=d_losses, shared_parameters=list(D.shared_parameters()),
                    task_specific_parameters=list(D.task_specific_parameters()))
        torch.cuda.synchronize()
    finally:
        ops.set_conv_mode("auto", 3)
        NW.set_dropout_mask_provider(None)
    _, g32 = oracle_d_grads(sd0, x.cpu(), y.cpu(), mk, 17, torch.float32)
    _, g64 = oracle_d_grads(sd0, x.cpu(), y.cpu(), mk, 17, torch.float64)
    names = set(O.d_task_specific_names())
    # per tensor: 1e-3, or 30x the oracle's own fp32-vs-fp64 gap where summation order alone moves a tensor more
    rows = sorted(((rel_err(p.grad, g32[k]), max(1e-3, 30 * rel_err(g32[k], g64[k])), k)
                   for k, p in D.named_parameters() if k in names), reverse=True)
    assert len(rows) == len(names)
    print("folded task-specific gradients (simt): median %.2e, worst %s"
          % (rows[len(rows) // 2][0], [(k, "%.2e" % e, "%.2e" % t) for e, t, k in rows[:5]]))
    assert rows[len(rows) // 2][0] <= 1e-4
    assert all(e <= t for e, t, _ in rows), [r for r in rows if r[0] > r[1]]
