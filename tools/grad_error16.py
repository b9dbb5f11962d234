#!/usr/bin/env python
"""Per-tensor rel-L2 of the parameter gradients of the fp16-storage training path against the fp32-storage path
(round-1 kernels) on the same rays / projections.

    python tools/grad_error16.py [n_rays] [seed|room]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import sinnerf_b200  # noqa: E402
from oracle import render_oracle as orc  # noqa: E402  (seeded weights only)
from sinnerf_b200 import synthetic  # noqa: E402
from sinnerf_b200.nerf import NeRF, Embedding  # noqa: E402
from sinnerf_b200.rendering import render_rays  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
which = sys.argv[2] if len(sys.argv) > 2 else "seed"
dev = torch.device("cuda:0")
if which == "room":
    z = np.load(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "room_weights.npz"))
    pc = {k[7:]: torch.from_numpy(z[k].copy()) for k in z.files if k.startswith("coarse/")}
    pf = {k[5:]: torch.from_numpy(z[k].copy()) for k in z.files if k.startswith("fine/")}
    rays = synthetic.random_rays("llff", n, seed=3)
else:
    pc, pf = orc.default_init_params(0), orc.default_init_params(1)
    rays = synthetic.random_rays("lego", n, seed=3)
emb = [Embedding(3, 10), Embedding(3, 4)]
g = torch.Generator().manual_seed(2)
rng = {"perturb_u": torch.rand(n, 64, generator=g), "noise_coarse": torch.randn(n, 64, generator=g),
       "pdf_u": torch.rand(n, 64, generator=g), "noise_fine": torch.randn(n, 128, generator=g)}
rng = {k: v.to(dev) for k, v in rng.items()}
grads, proj = {}, None
for storage in ("fp32", "fp16"):
    sinnerf_b200.set_train_storage(storage)
    models = []
    for p in (pc, pf):
        m = NeRF(use_new_activation=True)
        m.load_state_dict(p)
        models.append(m.to(dev))
    out = render_rays(models, emb, rays.to(dev), 64, False, 1.0, 1.0, 64, 32768, False, _rng=rng)
    if proj is None:
        gp = torch.Generator().manual_seed(5)
        proj = {k: torch.randn(v.shape, generator=gp).to(dev) for k, v in out.items()}
    sum((out[k] * proj[k]).sum() for k in proj).backward()
    grads[storage] = [{k: p.grad.detach().double().cpu() for k, p in m.named_parameters()} for m in models]
print(f"{which} weights, {n} rays: rel-L2 of fp16-storage gradients vs fp32-storage")
for name, a, b in (("coarse", grads["fp16"][0], grads["fp32"][0]), ("fine", grads["fp16"][1], grads["fp32"][1])):
    for k in a:
        nb = float(b[k].norm())
        if nb == 0:
            continue
        print(f"  {name:6s} {k:28s} {float((a[k] - b[k]).norm()) / nb:.2e}")
