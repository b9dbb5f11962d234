"""Randomised differential test: the CPU oracle against the REFERENCE ITSELF.

The reference's results on these inputs were recorded by running it (tests/golden/make_golden.py
reference_cases -> tests/golden/reference_cases.npz); the oracle is run here and compared with them.
Seeds, sizes and option combinations beyond the other goldens: use_disp, white_back, perturb/noise (the
reference draws from the global generator in the order rand, randn, rand, randn -- the oracle must consume it
identically), N_importance = 0, test_time.
"""
import zlib

import numpy as np
import pytest
import torch

from oracle import render_oracle as orc
from tests._common import load_npz

# gradient tensors with more entries than this are stored as norm + sample + projections (keeps the golden small)
GRAD_FULL_MAX = 768
GRAD_SAMPLE = 1024
GRAD_PROJECTIONS = 16


def grad_probe(numel, key):
    """(entry indices, (numel, GRAD_PROJECTIONS) N(0, 1) projection matrix) for the parameter tensor `key`, seeded by
    its name."""
    g = torch.Generator().manual_seed(zlib.crc32(key.encode()))
    return (torch.randperm(numel, generator=g)[:GRAD_SAMPLE],
            torch.randn(numel, GRAD_PROJECTIONS, generator=g, dtype=torch.float64))


@pytest.fixture(scope="module")
def gold():
    return load_npz("reference_cases.npz")


def t(x):
    return torch.from_numpy(np.asarray(x).copy())


def outputs(gold, prefix):
    return {k[len(prefix):]: t(v) for k, v in gold.items() if k.startswith(prefix)}


CASES = [
    # shape, n, S, Ni, use_disp, perturb, noise_std, white_back, seed
    ("lego", 33, 64, 64, False, 0.0, 0.0, True, 1),
    ("llff", 20, 48, 24, False, 1.0, 1.0, False, 2),
    ("dtu", 17, 32, 16, True, 1.0, 0.0, True, 3),
    ("lego", 9, 64, 0, False, 0.0, 1.0, False, 4),
    ("llff", 5, 16, 40, True, 0.0, 0.0, False, 5),
]


@pytest.mark.parametrize("shape,n,S,Ni,use_disp,perturb,noise_std,white_back,seed", CASES)
def test_render_rays_oracle_equals_live_reference(gold, shape, n, S, Ni, use_disp, perturb, noise_std, white_back, seed):
    i = CASES.index((shape, n, S, Ni, use_disp, perturb, noise_std, white_back, seed))
    assert gold[f"render{i}_cfg"].tolist() == [n, S, Ni, use_disp, perturb, noise_std, white_back, seed]
    rays = t(gold[f"render{i}_rays"])
    pc, pf = orc.default_init_params(10 + seed), orc.default_init_params(20 + seed)
    want = outputs(gold, f"render{i}_out_")
    with torch.no_grad():
        torch.manual_seed(100 + seed)
        got = orc.render_rays(pc, pf if Ni > 0 else None, rays, N_samples=S, N_importance=Ni, use_disp=use_disp, perturb=perturb,
                              noise_std=noise_std, white_back=white_back)
    assert want
    for k, v in want.items():
        assert k in got, k
        assert got[k].shape == v.shape, k
        err = float((got[k] - v).abs().max())
        scale = max(float(v.abs().max()), 1e-6)
        assert err <= 2e-5 * scale, (k, err, scale)


def test_test_time_keys_and_values(gold):
    rays = t(gold["testtime_rays"])
    pc, pf = orc.default_init_params(1), orc.default_init_params(2)
    want = outputs(gold, "testtime_out_")
    with torch.no_grad():
        got = orc.render_rays(pc, pf, rays, N_samples=64, N_importance=64, noise_std=0.0, white_back=True, test_time=True)
    assert set(k for k in got if not k.startswith("_")) == set(want)
    for k, v in want.items():
        assert float((got[k] - v).abs().max()) <= 2e-5 * max(float(v.abs().max()), 1e-6), k


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_sample_pdf_oracle_equals_live_reference(gold, seed):
    bins, w = t(gold[f"pdf{seed}_bins"]), t(gold[f"pdf{seed}_w"])
    assert float(w[0].abs().sum()) == 0.0              # all-zero weights row (the eps path)
    want = t(gold[f"pdf{seed}_out"])
    got = orc.sample_pdf(bins, w, want.shape[1], det=True)
    # identical arithmetic; allow the inverse-CDF's knot discontinuity (SURVEY hard part 3) on a few samples
    diff = (got - want).abs()
    assert float(diff.median()) == 0.0
    assert int((diff > 1e-5).sum()) <= 4


def test_autograd_oracle_equals_live_reference(gold):
    """Gradients of a random projection of all outputs w.r.t. all 48 parameter tensors: reference autograd vs
    autograd through the oracle (perturb and noise on: the sample_pdf detach and the RNG order both matter).
    Small tensors are compared whole; for the large ones the golden keeps the gradient's norm, a seeded sample of
    its entries and its dot products with seeded N(0, 1) vectors p: E[<a - b, p>^2] = |a - b|^2, so the RMS of the
    projected differences estimates the whole tensor's error and is held to the same bar."""
    rays = t(gold["grad_rays"])
    pc, pf = orc.default_init_params(31), orc.default_init_params(32)
    oc = {k: v.clone().requires_grad_(True) for k, v in pc.items()}
    of = {k: v.clone().requires_grad_(True) for k, v in pf.items()}
    proj = outputs(gold, "grad_proj_")
    torch.manual_seed(77)
    got = orc.render_rays(oc, of, rays, N_samples=32, N_importance=24, perturb=1.0, noise_std=1.0, white_back=False)
    sum((got[k] * proj[k]).sum() for k in proj).backward()
    ref_none = set(gold["grad_none"].tolist())
    n_checked = 0
    for which, params in (("coarse", oc), ("fine", of)):
        for k, v in params.items():
            key = f"{which}/{k}"
            a, b_none = v.grad, key in ref_none
            if a is None or b_none:
                # a gradient only one side has must be zero
                assert (a is None or float(a.abs().sum()) == 0.0) and (b_none or float(gold[f"gnorm_{key}"]) == 0.0), key
                continue
            a = a.double().flatten()
            b_norm = max(float(gold[f"gnorm_{key}"]), 1e-12)
            assert abs(float(a.norm()) - b_norm) <= 2e-4 * b_norm, (key, float(a.norm()), b_norm)
            if f"grad_{key}" in gold:
                b = t(gold[f"grad_{key}"]).double().flatten()
                assert float((a - b).norm()) <= 2e-4 * b_norm, (key, float((a - b).norm()) / b_norm)
            else:
                idx, p = grad_probe(a.numel(), key)
                b = t(gold[f"gsample_{key}"]).double()
                assert float((a[idx] - b).norm()) <= 2e-4 * max(float(b.norm()), 1e-12), key
                rms = float((a @ p - t(gold[f"gproj_{key}"])).square().mean().sqrt())
                assert rms <= 2e-4 * b_norm, (key, rms / b_norm)
            n_checked += 1
    assert n_checked + len(ref_none) == 48
