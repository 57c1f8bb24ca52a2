"""Parity at BASELINE.json's full sizes, where the driver's `-m gpu` run sees it: the north-star point
(131 072 / 512^2), LaRa's own Gaussian count (524 288 / 512^2) and configs[3] (262 144 / 1024^2), all
against what the UNMODIFIED reference computes on a B200 (tests/golden/reference) -- integer state, colour and
aux maps bit for bit, gradients on a seeded sample within 1e-4 (or 10x the reference's own run-to-run atomic
noise) -- plus a fixed-seed 25-configuration slice of tools/parity_sweep.py (ragged sizes, SH degrees 0-3, needle splats,
saturated scenes, cameras inside the cloud)."""
import numpy as np
import pytest
import torch

from helpers import Reference, run_candidate, tile_pixel_mask

pytestmark = pytest.mark.gpu

HEADLINE = [  # P, size, seed
    (131072, 512, 0),
    (524288, 512, 1),
    (262144, 1024, 2),
]
SWEEP_SEED = 20260924
GRAD_KEYS = (("g_means3D", "means3D"), ("g_sh", "shs"), ("g_opacities", "opacities"), ("g_scales", "scales"),
             ("g_rotations", "rotations"))


def _compare(mine, r, H, W, prefix="", with_noise=False):
    """Names of what differs from the reference's stored outputs `r` (keys under `prefix`), and the worst gradient error."""
    errs = []

    def chk(name, ok):
        if not ok:
            errs.append(name)
    p = prefix
    chk("radii", r.equal(p + "radii", mine["radii"]))
    chk("num_rendered", mine["num_rendered"] == r[p + "num_rendered"])
    if mine["num_rendered"] == r[p + "num_rendered"]:
        chk("point_list", r.equal(p + "point_list", mine["point_list"]))
    chk("ranges", r.equal(p + "ranges", mine["ranges"]))
    chk("n_contrib", r.equal(p + "n_contrib", mine["n_contrib"][0]))
    m = tile_pixel_mask(mine["ranges"], H, W)
    chk("median_contributor", r.equal(p + "median_contributor", mine["n_contrib"][1][m]))
    chk("color", r.equal(p + "color", mine["color"]))
    chk("allmap", r.equal(p + "allmap", mine["allmap"]))
    chk("accum", r.equal(p + "accum", mine["accum"]))
    worst = 0.0
    for a_, b_ in GRAD_KEYS:
        e = r.rel_err(p + b_, mine[a_])
        noise = r[p + "noise." + b_] if with_noise else 0.0
        worst = max(worst, e)
        chk(f"grad_{b_}({e:.1e}, ref noise {noise:.1e})", np.isfinite(mine[a_]).all() and e < max(1e-4, 10 * noise))
    return errs, worst


@pytest.mark.parametrize("P,size,seed", HEADLINE)
def test_headline_sizes_vs_reference(cuda_device, P, size, seed):
    from lara_b200 import scene as S
    sc = S.scene(P, seed, sh_degree=1)
    cam = S.cameras(3, size, size, seed)[seed % 3]
    bg = torch.ones(3)
    gc, ga = S.upstream_grads(size, size, seed)
    mine = run_candidate(sc, cam, bg, cuda_device, grads=(gc, ga))
    errs, worst = _compare(mine, Reference(f"headline-{P}_{size}_s{seed}"), size, size, with_noise=True)
    assert not errs, (errs, worst)
    assert mine["num_rendered"] > P          # the configuration really has LaRa-like overdraw


def _sweep_config(rng):
    from lara_b200 import scene as S
    P = int(rng.choice([500, 3000, 20000, 60000, 150000, 300000]))
    H = int(rng.choice([64, 100, 200, 256, 333, 512, 768])); W = int(rng.choice([64, 120, 200, 256, 400, 512, 700]))
    deg = int(rng.integers(0, 4)); bgv = float(rng.choice([0.0, 0.5, 1.0])); seed = int(rng.integers(0, 10000))
    sc = S.scene(P, seed, sh_degree=deg)
    sc["scales"] = sc["scales"] * float(rng.choice([0.3, 1.0, 2.5, 6.0]))
    if rng.random() < 0.3:
        sc["scales"][:, 1] *= 0.05                      # needle-like splats (edge-on conics)
    if rng.random() < 0.3:
        sc["opacities"] = torch.rand(sc["opacities"].shape, generator=torch.Generator().manual_seed(seed))  # saturation
    fov = float(rng.choice([0.4, 0.75, 1.3])); radius = float(rng.choice([0.9, 1.905, 4.0]))   # 0.9: camera inside the cloud
    cam = S.cameras(3, H, W, seed, fov=fov, radius=radius)[seed % 3]
    return dict(P=P, H=H, W=W, deg=deg, bg=bgv, seed=seed, fov=fov, radius=radius), sc, cam


def test_parity_sweep_slice_25_configurations(cuda_device):
    from lara_b200 import scene as S
    rng = np.random.default_rng(SWEEP_SEED)
    ref = Reference("sweep25")
    failures, worst = [], 0.0
    for it in range(25):
        tag, sc, cam = _sweep_config(rng)
        bg = torch.full((3,), tag["bg"])
        gc, ga = S.upstream_grads(tag["H"], tag["W"], tag["seed"])
        mine = run_candidate(sc, cam, bg, cuda_device, grads=(gc, ga))
        errs, w = _compare(mine, ref, tag["H"], tag["W"], prefix=f"{it}/")
        worst = max(worst, w)
        if errs:
            failures.append((tag, errs))
    assert not failures, (failures, worst)
