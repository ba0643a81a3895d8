"""Generates the golden fixtures under tests/golden/ from the LIVE reference, on CPU.

Run:   MTDGAN_REFERENCE=<checkout of babbu3682/MTD-GAN> CUDA_VISIBLE_DEVICES="" python tests/golden/make_golden.py
The fixtures travel with the repo, so the tests need no copy of the reference.
"""
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import torch  # noqa: E402

from _golden_util import save, summarize  # noqa: E402
from _refload import load_reference  # noqa: E402
from oracle import mtdgan_oracle as O  # noqa: E402

torch.set_num_threads(os.cpu_count())
ref = load_reference()
N = ref.networks


class MaskDrop(torch.nn.Module):
    """Stand-in for nn.Dropout(0.3) that multiplies by pre-drawn (already scaled) masks, in call order."""

    def __init__(self, masks):
        super().__init__()
        self.masks, self.p = list(masks), 0.3

    def forward(self, x):
        return x * self.masks.pop(0) if self.training else x


def drop_mask(b, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, 512, generator=g) >= 0.3).float() / 0.7


def seeded_model():
    torch.manual_seed(2024)
    random.seed(2024)
    return N.MTD_GAN_Method()


# 1. initial state fingerprint ------------------------------------------------------------------
m = seeded_model()
save("state_summary.pt", {k: summarize(v, 8) for k, v in m.state_dict().items()})

# 2/3. generator forward --------------------------------------------------------------------------
m.eval()
with torch.no_grad():
    x64 = O.synthetic_pair(2, 64, seed=11)[0]
    save("gen_fwd_64.pt", {"out": m.Generator(x64)})
    x512 = O.synthetic_pair(1, 512, seed=12)[0]
    save("gen_fwd_512.pt", {"out": m.Generator(x512)})            # fp32 storage (1 MiB): compared at 1e-4

# 4. stand-alone FFT_ConvBlock forward + backward ---------------------------------------------------
torch.manual_seed(5)
blk = N.FFT_ConvBlock(32)
g = torch.Generator().manual_seed(6)
xb = (0.5 * torch.randn(1, 32, 64, 64, generator=g)).requires_grad_(True)
wgt = torch.randn(1, 32, 64, 64, generator=g)
out = blk(xb)
(out * wgt).sum().backward()
save("fftblock_64.pt", {"out": out.detach(), "grads": {k: p.grad.clone() for k, p in blk.named_parameters()}})
save("fftblock_64_dx.pt", {"dx": xb.grad})                       # a file of its own: each stays under 1 MB

# 5. discriminator: train-mode forward/backward with an injected dropout mask, then eval ----------
m = seeded_model()
D = m.Discriminator
yb = O.synthetic_pair(2, 64, seed=13)[1]
D.train()
D.c_drop = MaskDrop([drop_mask(2, 14)])
enc, dec, rec = D(yb)
g = torch.Generator().manual_seed(15)
a, b, c = torch.randn(enc.shape, generator=g), torch.randn(dec.shape, generator=g), torch.randn(rec.shape, generator=g)
((enc * a).sum() + (dec * b).sum() / 64 + (rec * c).sum() / 64).backward()
fix = {"enc": enc.detach(), "dec": dec.detach(), "rec": rec.detach(),
       "grads": {k: summarize(p.grad) for k, p in D.named_parameters() if p.grad is not None},
       "buffers": {k: summarize(v, 8) for k, v in D.named_buffers()}}
D.eval()
with torch.no_grad():
    e2, d2, r2 = D(yb)
fix.update({"eval_enc": e2, "eval_dec": d2, "eval_rec": r2})
save("disc_64.pt", fix)

# 6. one full training step, B = 4 (BASELINE configs[0]) -------------------------------------------
m = seeded_model()
m.train()
m.Discriminator.c_drop = MaskDrop([drop_mask(4, 21 + i) for i in range(5)])
x, y = O.synthetic_pair(4, 64, seed=1234)
Dn = m.Discriminator
opt_D = torch.optim.AdamW(Dn.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4)
opt_G = torch.optim.AdamW(m.Generator.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4)
wm = ref.weight_methods.WeightMethods('pcgrad', n_tasks=3, device=torch.device('cpu'))
random.seed(99)
opt_D.zero_grad(); Dn.zero_grad()
d_losses, d_det = m.d_loss(x, y)
shared = list(Dn.shared_parameters())
per_task = [torch.autograd.grad(l, shared, retain_graph=True) for l in d_losses]
flat = [torch.cat([t.flatten() for t in tg]).double() for tg in per_task]
gram = torch.tensor([[float(p @ q) for q in flat] for p in flat], dtype=torch.float64)
random.seed(99)
wm.backward(losses=d_losses, shared_parameters=shared, task_specific_parameters=list(Dn.task_specific_parameters()),
            last_shared_parameters=list(Dn.last_shared_parameters()))
step = {"d_losses": d_losses.detach(), "d_details": {k: v.detach() for k, v in d_det.items()}, "gram": gram,
        "per_task_norms": [float(f.norm()) for f in flat],
        "d_grads": {k: (summarize(p.grad) if p.grad is not None else None) for k, p in Dn.named_parameters()}}
opt_D.step()
opt_G.zero_grad(); m.Generator.zero_grad()
g_loss, g_det = m.g_loss(x, y)
g_loss.backward()
step.update({"g_loss": g_loss.detach(), "g_details": {k: v.detach() for k, v in g_det.items()},
             "g_grads": {k: summarize(p.grad) for k, p in m.Generator.named_parameters()}})
opt_G.step()
step["state_after"] = {k: summarize(v, 8) for k, v in m.state_dict().items()}

# fp32-vs-fp64 gap of the REFERENCE itself on the same weights/inputs/masks: the conditioning noise floor of
# every gradient (ReLU-mask flips at near-zero pre-activations make some sums non-reproducible below ~1e-2)
m64 = seeded_model().double()
m64.train()
m64.edge_loss.kernel = m64.edge_loss.kernel.double()
m64.Discriminator.c_drop = MaskDrop([drop_mask(4, 21 + i).double() for i in range(5)])
x64, y64 = x.double(), y.double()
D64 = m64.Discriminator
opt_D64 = torch.optim.AdamW(D64.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4)
random.seed(99)
dl64, _ = m64.d_loss(x64, y64)
wm.backward(losses=dl64, shared_parameters=list(D64.shared_parameters()),
            task_specific_parameters=list(D64.task_specific_parameters()),
            last_shared_parameters=list(D64.last_shared_parameters()))


def gap(g32, g64):
    a, b = g32.detach().double().flatten(), g64.detach().double().flatten()
    rms = float(b.norm()) / (b.numel() ** 0.5) + 1e-300
    return {"norm": abs(float(a.norm()) - float(b.norm())) / (float(b.norm()) + 1e-300), "samp": float((a - b).abs().max()) / rms}


d32 = {k: p.grad for k, p in Dn.named_parameters()}
# note: Dn grads were overwritten by the G step's backward (dead accumulation); recompute the D-step fp32 grads
m32 = seeded_model(); m32.train()
m32.Discriminator.c_drop = MaskDrop([drop_mask(4, 21 + i) for i in range(5)])
random.seed(99)
dl32, _ = m32.d_loss(x, y)
wm.backward(losses=dl32, shared_parameters=list(m32.Discriminator.shared_parameters()),
            task_specific_parameters=list(m32.Discriminator.task_specific_parameters()),
            last_shared_parameters=list(m32.Discriminator.last_shared_parameters()))
step["d_grads_noise"] = {k: gap(p.grad, dict(D64.named_parameters())[k].grad) for k, p in m32.Discriminator.named_parameters()
                         if p.grad is not None}
opt_D64.step()
torch.optim.AdamW(m32.Discriminator.parameters(), lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-4).step()
gl64, _ = m64.g_loss(x64, y64)
gl64.backward()
gl32, _ = m32.g_loss(x, y)
gl32.backward()
step["g_grads_noise"] = {k: gap(p.grad, dict(m64.Generator.named_parameters())[k].grad)
                         for k, p in m32.Generator.named_parameters()}
print("worst D noise", max(v["samp"] for v in step["d_grads_noise"].values()),
      "worst G noise", max(v["samp"] for v in step["g_grads_noise"].values()))
save("train_step_b4.pt", step)

# 7. loss terms: values, gradients, NDS mask with special values ------------------------------------
g = torch.Generator().manual_seed(31)
xs, ys = O.synthetic_pair(4, 64, seed=32)
pred = torch.rand(4, 1, 64, 64, generator=g).requires_grad_(True)
spec = xs.clone()
spec.view(-1)[:6] = torch.tensor([0.0, -0.0, 1e-42, float("nan"), 1.0, 0.5])
ysp = ys.clone()
ysp.view(-1)[:6] = torch.tensor([-0.0, 0.0, 0.0, 0.3, 1.0, 0.5 + 2 ** -24])
lf = {}
for name, fn in (("ls_gan1", lambda p: ref.losses.ls_gan(p, 1.0)), ("nds0", lambda p: ref.losses.NDS_Loss(p, 0.0, xs - ys)),
                 ("charb", lambda p: ref.losses.CharbonnierLoss()(p, ys)), ("edge", lambda p: ref.losses.EdgeLoss()(p, ys))):
    pred.grad = None
    v = fn(pred)
    v.backward()
    lf[name] = {"value": v.detach(), "grad": pred.grad.clone()}
lf["pred"] = pred.detach()
lf["mask_special"] = torch.abs(spec - ysp).bool()
lf["spec"], lf["ysp"] = spec, ysp
save("losses.pt", lf)

# 8. the reference's only known-answer vector: module/pcgrad.py demo (seed 4) -----------------------
P = ref.pcgrad
demo = []
for cls, heads in ((P.TestNet, False), (P.MultiHeadTestNet, True)):
    torch.manual_seed(4)
    xd, yd = torch.randn(2, 3), torch.randn(2, 4)
    net = cls()
    pc = P.PCGrad(torch.optim.Adam(net.parameters()))
    pc.zero_grad()
    if heads:
        y1, y2 = net(xd)
        l1, l2 = torch.nn.MSELoss()(y1, yd), torch.nn.MSELoss()(y2, yd)
    else:
        yp = net(xd)
        l1, l2 = torch.nn.L1Loss()(yp, yd), torch.nn.MSELoss()(yp, yd)
    pc.pc_backward([l1, l2])
    demo.append([p.grad.clone() for p in net.parameters()])
save("pcgrad_demo.pt", {"grads": demo})
print("done")
