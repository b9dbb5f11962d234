#!/usr/bin/env python
"""Generate the committed golden fixtures by running the REFERENCE itself.

Needs a checkout of the original SinNeRF repository (models/, datasets/, ckpts/room.ckpt):

    SINNERF_REF=/path/to/SinNeRF python tests/golden/make_golden.py

Imports the reference's own ``models/rendering.py``, ``models/nerf.py``
(unmodified) on CPU/fp32 and records inputs + outputs of
every stage of the hot path.  Nothing here is used at run time by the product;
tests compare (a) the oracle and (b) the CUDA path against these files.

Outputs (tests/golden/):
  room_weights.npz   the reference's trained checkpoint ckpts/room.ckpt re-saved
                     as plain arrays (realistic weight statistics; SURVEY.md 2 #15)
  stages.npz         Embedding / NeRF.forward / sample_pdf / activations goldens
  render_*.npz       whole render_rays cases (rays, config, RNG tensors, outputs)
  reference_cases.npz  the randomised cases of tests/test_oracle_vs_reference_live.py
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("SINNERF_REF", "")
if not os.path.isdir(os.path.join(REF, "models")):
    sys.exit("set SINNERF_REF to a checkout of the original SinNeRF repository")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REF)
sys.path.insert(1, ROOT)

from models.nerf import NeRF, Embedding            # noqa: E402  (reference)
from models.rendering import render_rays, sample_pdf  # noqa: E402  (reference)
from models.activations import shifted_softplus, widened_sigmoid  # noqa: E402

from sinnerf_b200 import synthetic                  # noqa: E402
from oracle.render_oracle import default_init_params  # noqa: E402

torch.set_num_threads(8)


def np_(t):
    return t.detach().cpu().numpy()


def load_room():
    sd = torch.load(os.path.join(REF, "ckpts/room.ckpt"), map_location="cpu", weights_only=True)
    out = {}
    for which in ("nerf_coarse", "nerf_fine"):
        for k, v in sd.items():
            if k.startswith(which + "."):
                out[which[5:] + "/" + k[len(which) + 1:]] = np_(v.float())
    return out


def model_from(params):
    m = NeRF(use_new_activation=True)
    m.load_state_dict({k: torch.as_tensor(v) for k, v in params.items()})
    return m.eval()


def seeded_models(seed):
    torch.manual_seed(seed)
    c = NeRF(use_new_activation=True)
    # check that the oracle's init helper reproduces the module's default init
    p = default_init_params(seed)
    for k, v in c.state_dict().items():
        assert torch.equal(v, p[k]), k
    torch.manual_seed(seed + 1)
    f = NeRF(use_new_activation=True)
    return c.eval(), f.eval()


def room_models(room):
    c = model_from({k[7:]: v for k, v in room.items() if k.startswith("coarse/")})
    f = model_from({k[5:]: v for k, v in room.items() if k.startswith("fine/")})
    return c, f


def replay_rng(seed, n, sc, ni, perturb):
    """The tensors render_rays draws, in its order (rendering.py:281,224,43,224)."""
    torch.manual_seed(seed)
    r = {}
    if perturb > 0:
        r["perturb_u"] = torch.rand(n, sc)
    r["noise_coarse"] = torch.randn(n, sc)
    if ni > 0:
        if perturb > 0:
            r["pdf_u"] = torch.rand(n, ni)
        r["noise_fine"] = torch.randn(n, sc + ni)
    return r


def render_case(name, models, rays, *, n_samples=64, n_importance=64, use_disp=False, perturb=0.0,
                noise_std=0.0, white_back=False, test_time=False, rng_seed=1234, weights_tag="seed0"):
    emb = [Embedding(3, 10), Embedding(3, 4)]
    with torch.no_grad():
        torch.manual_seed(rng_seed)
        res = render_rays(models, emb, rays, n_samples, use_disp, perturb, noise_std, n_importance,
                          1024 * 32, white_back, test_time=test_time)
    rng = replay_rng(rng_seed, rays.shape[0], n_samples, n_importance, perturb)
    out = {"rays": np_(rays),
           "cfg": np.array([n_samples, n_importance, int(use_disp), perturb, noise_std, int(white_back),
                            int(test_time)], dtype=np.float64),
           "weights_tag": np.array(weights_tag)}
    for k, v in res.items():
        out["out_" + k] = np_(v)
    for k, v in rng.items():
        out["rng_" + k] = np_(v)
    path = os.path.join(HERE, f"render_{name}.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items() if k.startswith("out_")})


def grad_golden(room):
    """Reference autograd: d(loss)/d(params) for a fixed random projection of all outputs.
    Stores per-tensor gradient norms and the full gradients of the small tensors."""
    trained = [m.train() for m in room_models(room)]
    rays = synthetic.random_rays("llff", 24, seed=5)
    emb = [Embedding(3, 10), Embedding(3, 4)]
    torch.manual_seed(4321)
    res = render_rays(trained, emb, rays, 64, False, 1.0, 1.0, 64, 1024 * 32, False)
    rng = replay_rng(4321, 24, 64, 64, 1.0)
    g = torch.Generator().manual_seed(11)
    proj = {k: torch.randn(v.shape, generator=g) for k, v in sorted(res.items())}
    loss = sum((res[k] * proj[k]).sum() for k in sorted(res))
    loss.backward()
    out = {"rays": np_(rays), "loss": np.array(float(loss))}
    for k, v in rng.items():
        out["rng_" + k] = np_(v)
    for k in sorted(proj):
        out["proj_" + k] = np_(proj[k])
    for which, m in (("coarse", trained[0]), ("fine", trained[1])):
        for name, prm in m.named_parameters():
            out[f"gnorm_{which}/{name}"] = np.array(float(prm.grad.norm()))
            if prm.numel() <= 768:
                out[f"grad_{which}/{name}"] = np_(prm.grad)
    path = os.path.join(HERE, "grad_llff_room_train.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "loss", float(loss))


def rays_golden():
    """Reference ray generation: datasets/ray_utils.py (blender/LLFF) and datasets/dtu_proj.py (DTU)."""
    from datasets.ray_utils import get_ray_directions, get_rays
    g = torch.Generator().manual_seed(21)
    out = {}
    for tag, (H, W, f) in {"lego": (40, 56, 77.7), "llff": (378 // 6, 504 // 6, 410.0 / 6)}.items():
        c2w = torch.cat([torch.linalg.qr(torch.randn(3, 3, generator=g))[0], torch.randn(3, 1, generator=g)], 1)
        d = get_ray_directions(H, W, f)
        o, dw = get_rays(d, c2w)
        near, far = 2.0, 6.0
        rays = torch.cat([o, dw, near * torch.ones_like(o[:, :1]), far * torch.ones_like(o[:, :1])], 1)
        out[f"{tag}_cfg"] = np.array([H, W, f, near, far])
        out[f"{tag}_c2w"] = np_(c2w)
        out[f"{tag}_rays"] = np_(rays)
    # DTU: own directions function (imports the dataset module lazily: it needs cv2 / PIL only for loading)
    H, W, fx, fy, cx, cy = 32, 40, 361.5, 360.9, 19.3, 16.8
    c2w = torch.cat([torch.linalg.qr(torch.randn(3, 3, generator=g))[0], torch.randn(3, 1, generator=g)], 1)
    try:
        from datasets.dtu_proj import get_ray_directions_dtu
        d = get_ray_directions_dtu(H, W, [fx, fy], [cx, cy])
    except Exception as e:   # module-level imports of dtu_proj that are missing here
        print("dtu_proj import failed (", e, "); using the formula of dtu_proj.py:31-32 via ray_utils.create_meshgrid")
        from datasets.ray_utils import create_meshgrid
        i, j = create_meshgrid(H, W, normalized_coordinates=False)[0].unbind(-1)
        d = torch.stack([(i - cx) / fx, (j - cy) / fy, torch.ones_like(i)], -1)
    o, dw = get_rays(d, c2w)
    rays = torch.cat([o, dw, 2.125 * torch.ones_like(o[:, :1]), 4.525 * torch.ones_like(o[:, :1])], 1)
    out["dtu_cfg"] = np.array([H, W, fx, fy, cx, cy, 2.125, 4.525])
    out["dtu_c2w"] = np_(c2w)
    out["dtu_rays"] = np_(rays)
    path = os.path.join(HERE, "rays.npz")
    np.savez_compressed(path, **out)
    print("wrote", path)


def c1_full():
    """BASELINE configs[0] in full: all 1 024 rays of the C1 case (the 128-ray prefix is render_c1_seed0_64p0)."""
    seed_models = list(seeded_models(0))
    render_case("c1_full_seed0_64p0", seed_models[:1], synthetic.random_rays("lego", 1024, seed=0),
                n_importance=0, white_back=False)


def reference_cases():
    """What tests/test_oracle_vs_reference_live.py compares the oracle with, on its inputs: render_rays of its
    randomised cases, the test_time keys, sample_pdf on random bins / weights, and reference autograd.  Gradient
    tensors above GRAD_FULL_MAX entries are kept as norm + seeded sample + seeded projections (file size)."""
    from tests.test_oracle_vs_reference_live import CASES, GRAD_FULL_MAX, grad_probe
    out = {}
    for i, (shape, n, S, Ni, use_disp, perturb, noise_std, white_back, seed) in enumerate(CASES):
        rays = synthetic.random_rays(shape, n, seed=seed)
        models = [model_from(default_init_params(10 + seed)), model_from(default_init_params(20 + seed))]
        emb = [Embedding(3, 10), Embedding(3, 4)]
        with torch.no_grad():
            torch.manual_seed(100 + seed)
            res = render_rays(models, emb, rays, S, use_disp, perturb, noise_std, Ni, 1024, white_back, test_time=False)
        out[f"render{i}_cfg"] = np.array([n, S, Ni, use_disp, perturb, noise_std, white_back, seed], dtype=np.float64)
        out[f"render{i}_rays"] = np_(rays)
        for k, v in res.items():
            out[f"render{i}_out_{k}"] = np_(v)

    rays = synthetic.random_rays("lego", 12, seed=9)
    models = [model_from(default_init_params(1)), model_from(default_init_params(2))]
    with torch.no_grad():
        res = render_rays(models, [Embedding(3, 10), Embedding(3, 4)], rays, 64, False, 0, 0, 64, 1024, True, test_time=True)
    out["testtime_rays"] = np_(rays)
    for k, v in res.items():
        out[f"testtime_out_{k}"] = np_(v)

    for seed in (0, 1, 2):
        g = torch.Generator().manual_seed(seed)
        n, m, ni = 19, 23 + seed, 31
        bins = torch.sort(torch.rand(n, m + 1, generator=g) * 4 + 2, dim=-1).values
        w = torch.rand(n, m, generator=g) ** 3
        w[0] = 0.0                                    # all-zero weights row (the eps path)
        out[f"pdf{seed}_bins"], out[f"pdf{seed}_w"] = np_(bins), np_(w)
        out[f"pdf{seed}_out"] = np_(sample_pdf(bins, w, ni, det=True))

    rays = synthetic.random_rays("llff", 14, seed=21)
    models = [model_from(default_init_params(31)).train(), model_from(default_init_params(32)).train()]
    torch.manual_seed(77)
    res = render_rays(models, [Embedding(3, 10), Embedding(3, 4)], rays, 32, False, 1.0, 1.0, 24, 1024, False, test_time=False)
    g = torch.Generator().manual_seed(5)
    proj = {k: torch.randn(v.shape, generator=g) for k, v in res.items()}
    sum((res[k] * proj[k]).sum() for k in res).backward()
    out["grad_rays"] = np_(rays)
    for k, v in proj.items():
        out[f"grad_proj_{k}"] = np_(v)
    none = []
    for which, m in (("coarse", models[0]), ("fine", models[1])):
        for name, prm in m.named_parameters():
            key = f"{which}/{name}"
            if prm.grad is None:
                none.append(key)
                continue
            gr = prm.grad.double().flatten()
            out[f"gnorm_{key}"] = np.array(float(gr.norm()))
            if gr.numel() <= GRAD_FULL_MAX:
                out[f"grad_{key}"] = np_(prm.grad)
            else:
                idx, p = grad_probe(gr.numel(), key)
                out[f"gsample_{key}"] = np_(prm.grad.flatten()[idx])
                out[f"gproj_{key}"] = np_(gr @ p)
    out["grad_none"] = np.array(none, dtype=str)
    path = os.path.join(HERE, "reference_cases.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, len(out), "arrays")


def main():
    if "--only-c1-full" in sys.argv:
        c1_full()
        return
    if "--reference-cases-only" in sys.argv:
        reference_cases()
        return
    room = load_room()
    if "--rays-only" in sys.argv:
        rays_golden()
        return
    if "--grad-only" in sys.argv:
        grad_golden(room)
        return
    np.savez_compressed(os.path.join(HERE, "room_weights.npz"), **room)
    print("room_weights:", len(room), "tensors")

    # ---------------- stage goldens ----------------
    g = torch.Generator().manual_seed(0)
    st = {}
    x = (torch.rand(96, 3, generator=g) - 0.5) * 8.0
    x[0] = torch.tensor([0.1, 0.2, 0.3])
    x[1] = torch.tensor([3.9, -3.9, 7.7])          # |512 x| ~ 4e3 rad (LLFF scale)
    st["embed_x"] = np_(x)
    st["embed_xyz_out"] = np_(Embedding(3, 10)(x))
    st["embed_dir_out"] = np_(Embedding(3, 4)(x))
    st["embed_L2_kat"] = np_(Embedding(3, 2)(torch.tensor([[0.1, 0.2, 0.3]])))

    a = torch.linspace(-30, 30, 241)
    a = torch.cat([a, torch.tensor([1.0, 0.999999, 1.000001, 222.0, -222.0])])
    st["act_x"] = np_(a)
    st["act_softplus"] = np_(shifted_softplus(a))
    st["act_wsigmoid"] = np_(widened_sigmoid(a))

    # NeRF.forward on embedded inputs, default-init and trained weights
    pts = (torch.rand(200, 3, generator=g) - 0.5) * 6.0
    dirs = torch.randn(200, 3, generator=g)
    feat = torch.cat([Embedding(3, 10)(pts), Embedding(3, 4)(dirs)], -1)
    st["mlp_in"] = np_(feat)
    mc, mf = seeded_models(0)
    rc, rf = room_models(room)
    with torch.no_grad():
        st["mlp_seed0_out"] = np_(mc(feat))
        st["mlp_seed0_sigma"] = np_(mc(feat[:, :63], sigma_only=True))
        st["mlp_room_coarse_out"] = np_(rc(feat))
        st["mlp_room_fine_out"] = np_(rf(feat))

    # sample_pdf: known-answer vectors of SURVEY 8c + random cases
    bins5 = torch.tensor([[0., 1., 2., 3., 4.]])
    for tag, w, n in (("ones", [1., 1., 1., 1.], 5), ("spike", [0., 0., 1., 0.], 5),
                      ("zero", [0., 0., 0., 0.], 5), ("ramp", [.1, .2, .3, .4], 8)):
        st[f"pdf_kat_{tag}"] = np_(sample_pdf(bins5, torch.tensor([w]), n, det=True))
    zc = torch.sort(torch.rand(64, 64, generator=g) * 4 + 2, -1)[0]
    zmid = 0.5 * (zc[:, :-1] + zc[:, 1:])
    w = torch.rand(64, 62, generator=g) ** 4
    w[3] = 0.0                      # all-zero weights row
    w[4, :] = 0.0
    w[4, 17] = 1.0                  # single spike
    u = torch.rand(64, 64, generator=g)
    st["pdf_bins"], st["pdf_w"], st["pdf_u"] = np_(zmid), np_(w), np_(u)
    st["pdf_det_out"] = np_(sample_pdf(zmid, w, 64, det=True))
    torch.manual_seed(99)
    st["pdf_rand_out"] = np_(sample_pdf(zmid, w, 64, det=False))
    torch.manual_seed(99)
    st["pdf_rand_u"] = np_(torch.rand(64, 64))
    np.savez_compressed(os.path.join(HERE, "stages.npz"), **st)
    print("wrote stages.npz", len(st))

    # ---------------- whole render_rays goldens ----------------
    seed_models = list(seeded_models(0))
    trained = list(room_models(room))
    lego = synthetic.random_rays("lego", 96, seed=0)
    llff = synthetic.random_rays("llff", 96, seed=1)
    dtu = synthetic.random_rays("dtu", 64, seed=2)

    # C1 shape: 64+0, default init, no noise (configs[0])
    render_case("c1_seed0_64p0", seed_models[:1], synthetic.random_rays("lego", 1024, seed=0)[:128],
                n_importance=0, white_back=False)
    render_case("lego_seed0_64p64_wb", seed_models, lego, white_back=True)
    render_case("llff_room_64p64", trained, llff, weights_tag="room")
    render_case("llff_room_64p64_train", trained, llff, perturb=1.0, noise_std=1.0, weights_tag="room")
    render_case("dtu_seed0_64p64_disp", seed_models, dtu, use_disp=True, white_back=True)
    render_case("lego_room_testtime", trained, lego[:48], test_time=True, weights_tag="room")
    render_case("lego_seed0_32p16_odd", seed_models, lego[:33], n_samples=32, n_importance=16,
                perturb=0.5, noise_std=0.3, white_back=True)
    grad_golden(room)
    rays_golden()
    c1_full()
    reference_cases()


if __name__ == "__main__":
    main()
