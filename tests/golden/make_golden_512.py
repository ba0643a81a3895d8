"""Regenerates tests/golden/gen_fwd_512.pt alone (fp32) from the LIVE reference on CPU — the same statement
as section 2/3 of make_golden.py, for when only this fixture changes.
Run:   MTDGAN_REFERENCE=<checkout of babbu3682/MTD-GAN> CUDA_VISIBLE_DEVICES="" python tests/golden/make_golden_512.py"""
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import torch  # noqa: E402

from _golden_util import save  # noqa: E402
from _refload import load_reference  # noqa: E402
from oracle import mtdgan_oracle as O  # noqa: E402

torch.set_num_threads(os.cpu_count())
N = load_reference().networks
torch.manual_seed(2024)
random.seed(2024)
m = N.MTD_GAN_Method().eval()
with torch.no_grad():
    out = m.Generator(O.synthetic_pair(1, 512, seed=12)[0])
save("gen_fwd_512.pt", {"out": out})
