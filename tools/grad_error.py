#!/usr/bin/env python
"""rel-L2 of every parameter gradient (CUDA path vs autograd through the CPU oracle with the CUDA path's
fine depths injected).  SINNERF_B200_PRECISION selects the forward.

    python tools/grad_error.py [n_rays] [weights: seed|room] [loss: sum|proj]
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from oracle import render_oracle as orc  # noqa: E402
from sinnerf_b200 import synthetic  # noqa: E402
from sinnerf_b200.nerf import NeRF, Embedding  # noqa: E402
from sinnerf_b200.rendering import render_rays  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
weights = sys.argv[2] if len(sys.argv) > 2 else "seed"
loss_kind = sys.argv[3] if len(sys.argv) > 3 else "sum"
dev = torch.device("cuda:0")
rays = synthetic.random_rays("lego", n, seed=3)
if weights == "room":
    from tests._common import room_params
    pc, pf = room_params("coarse"), room_params("fine")
else:
    pc, pf = orc.default_init_params(0), orc.default_init_params(1)
models = []
for p in (pc, pf):
    m = NeRF(use_new_activation=True)
    m.load_state_dict(p)
    models.append(m.to(dev))
emb = [Embedding(3, 10), Embedding(3, 4)]
g = torch.Generator().manual_seed(5)


def loss_of(o, proj):
    keys = ("rgb_fine", "depth_fine", "rgb_coarse")
    if loss_kind == "sum":
        return sum(o[k].sum() for k in keys)
    return sum((o[k] * proj[k].to(o[k].device)).sum() for k in keys)


out = render_rays(models, emb, rays.to(dev), 64, False, 0, 0, 64, 32768, True, _return_intermediates=True)
proj = {k: torch.randn(out[k].shape, generator=g) for k in ("rgb_fine", "depth_fine", "rgb_coarse")}
loss_of(out, proj).backward()
oc = {k: v.clone().requires_grad_(True) for k, v in pc.items()}
of = {k: v.clone().requires_grad_(True) for k, v in pf.items()}
ref = orc.render_rays(oc, of, rays, N_samples=64, N_importance=64, noise_std=0.0, white_back=True,
                      z_fine_override=out["_inter"]["z_fine"].detach().cpu())
loss_of(ref, proj).backward()
print(f"n_rays={n} weights={weights} loss={loss_kind} "
      f"precision={os.environ.get('SINNERF_B200_PRECISION', 'default')}")
for name, ref_p, model in (("coarse", oc, models[0]), ("fine", of, models[1])):
    got = dict(model.named_parameters())
    row = []
    for k, v in ref_p.items():
        if float(v.grad.norm()) == 0.0:
            continue
        err = float((got[k].grad.double().cpu() - v.grad.double()).norm() / v.grad.double().norm())
        row.append(f"{k.replace('xyz_encoding_', 'L').replace('.weight', '.w').replace('.bias', '.b')}={err:.1e}")
    print(f"  {name}: " + " ".join(row))
