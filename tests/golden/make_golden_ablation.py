"""Golden fixtures for the ablation rows (SURVEY §8f-3) from the LIVE reference on CPU: for each of the ten
`Ablation_*` classes (arch/Ours/networks.py:1324-1936) the initial-state fingerprint, `d_loss` / `g_loss` totals and
details on 2 synthetic patches with injected dropout masks, and fingerprints of the gradients `d_loss.backward()` /
`g_loss.backward()` leave (engine.py:58-73).
Run:  MTDGAN_REFERENCE=<checkout of babbu3682/MTD-GAN> CUDA_VISIBLE_DEVICES="" python tests/golden/make_golden_ablation.py"""
import contextlib
import io
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
N = load_reference().networks
NAMES = ["Ablation_CLS", "Ablation_SEG", "Ablation_CLS_SEG", "Ablation_CLS_REC", "Ablation_SEG_REC", "Ablation_CLS_SEG_REC",
         "Ablation_CLS_SEG_REC_NDS", "Ablation_CLS_SEG_REC_RC", "Ablation_CLS_SEG_REC_NDS_RC",
         "Ablation_CLS_SEG_REC_NDS_RC_ResFFT"]


class MaskDrop(torch.nn.Module):
    def __init__(self, masks):
        super().__init__()
        self.masks, self.p = list(masks), 0.3

    def forward(self, x):
        return x * self.masks.pop(0) if self.training else x


def drop_mask(b, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(b, 512, generator=g) >= 0.3).float() / 0.7


def gap(g32, g64):
    """fp32-vs-fp64 gap of the REFERENCE itself (same method as make_golden.py): the conditioning noise floor of a
    gradient tensor (ReLU / LeakyReLU mask flips at near-zero pre-activations)."""
    a, b = g32.detach().double().flatten(), g64.detach().double().flatten()
    rms = float(b.norm()) / (b.numel() ** 0.5) + 1e-300
    return {"norm": abs(float(a.norm()) - float(b.norm())) / (float(b.norm()) + 1e-300), "samp": float((a - b).abs().max()) / rms}


def run64(name):
    """The same two backward passes in float64."""
    torch.manual_seed(2024)
    random.seed(2024)
    m = getattr(N, name)().double().train()
    m.edge_loss.kernel = m.edge_loss.kernel.double()
    if hasattr(m.Discriminator, "c_drop"):
        m.Discriminator.c_drop = MaskDrop([drop_mask(2, 900 + i).double() for i in range(5)])
    with contextlib.redirect_stdout(io.StringIO()):
        d_total, _ = m.d_loss(x.double(), y.double())
    d_total.backward()
    dg = {k: (None if p.grad is None else p.grad.clone()) for k, p in m.Discriminator.named_parameters()}
    m.zero_grad(set_to_none=True)
    with contextlib.redirect_stdout(io.StringIO()):
        g_total, _ = m.g_loss(x.double(), y.double())
    g_total.backward()
    return dg, {k: p.grad.clone() for k, p in m.Generator.named_parameters()}


out = {}
x, y = O.synthetic_pair(2, 64, seed=77)
for name in NAMES:
    torch.manual_seed(2024)
    random.seed(2024)
    m = getattr(N, name)().train()
    fix = {"state": {k: summarize(v, 8) for k, v in m.state_dict().items()}}
    if hasattr(m.Discriminator, "c_drop"):
        m.Discriminator.c_drop = MaskDrop([drop_mask(2, 900 + i) for i in range(5)])
    with contextlib.redirect_stdout(io.StringIO()):          # the reference prints tensor maxima
        d_total, d_det = m.d_loss(x, y)
    d_total.backward()
    dg64, gg64 = run64(name)
    fix["d_grads_noise"] = {k: gap(p.grad, dg64[k]) for k, p in m.Discriminator.named_parameters() if p.grad is not None}
    fix["d_total"] = float(d_total)
    fix["d_details"] = {k: float(v) for k, v in d_det.items()}
    fix["d_grads"] = {k: (None if p.grad is None else summarize(p.grad, 16)) for k, p in m.Discriminator.named_parameters()}
    m.zero_grad(set_to_none=True)
    with contextlib.redirect_stdout(io.StringIO()):
        g_total, g_det = m.g_loss(x, y)
    g_total.backward()
    fix["g_total"] = float(g_total)
    fix["g_details"] = {k: float(v) for k, v in g_det.items()}
    fix["g_grads"] = {k: summarize(p.grad, 16) for k, p in m.Generator.named_parameters()}
    fix["g_grads_noise"] = {k: gap(p.grad, gg64[k]) for k, p in m.Generator.named_parameters()}
    fix["buffers"] = {k: summarize(v, 8) for k, v in m.Discriminator.named_buffers()}
    out[name] = fix
    print(name, fix["d_total"], fix["g_total"], len(fix["d_grads"]), "worst D noise %.2e, worst G noise %.2e"
          % (max(v["samp"] for v in fix["d_grads_noise"].values()), max(v["samp"] for v in fix["g_grads_noise"].values())), flush=True)

# stand-alone REDCNN_Generator forward (eval)
torch.manual_seed(2024)
G = N.REDCNN_Generator(in_channels=1, out_channels=32, num_layers=10, kernel_size=3, padding=1).eval()
with torch.no_grad():
    out["redcnn_fwd_64"] = G(O.synthetic_pair(2, 64, seed=11)[0])
save("ablation.pt", out)
