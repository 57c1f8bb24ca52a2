"""Edge cases of the hot path on the GPU (the reference has no tests; these cover the cases
SURVEY.md section 7 lists): empty input, everything culled, one splat covering every tile,
thousands of instances in one tile (shared-memory and global sort paths), tied depths,
extreme opacities, saturated pixels, capacity overflow re-run, precomputed colours,
markVisible, non-contiguous inputs."""
import numpy as np
import pytest
import torch

from helpers import Reference, run_candidate, to_dev

pytestmark = pytest.mark.gpu


def _api(dev, sc, cam, bg, **kw):
    import diff_surfel_rasterization as DSR
    from lara_b200 import scene as S
    st = S.settings_for(cam, bg, sc["sh_degree"], dev, DSR.GaussianRasterizationSettings)
    return DSR, st, DSR.GaussianRasterizer(raster_settings=st)


def test_empty_scene_returns_zero_images(cuda_device):
    from lara_b200 import scene as S
    cam = S.cameras(1, 64, 64, 0)[0]
    sc = {k: v[:0] for k, v in S.scene(8, 0).items() if isinstance(v, torch.Tensor)}
    sc["sh_degree"] = 1
    scd = to_dev(sc, cuda_device)
    DSR, st, rast = _api(cuda_device, sc, cam, torch.ones(3))
    m3 = scd["means3D"].requires_grad_(True)
    color, radii, allmap = rast(means3D=m3, means2D=torch.zeros_like(m3), shs=scd["shs"], opacities=scd["opacities"],
                                scales=scd["scales"], rotations=scd["rotations"])
    # reference: zero-filled outputs when P == 0 (rasterize_points.cu:92-105), not background
    assert float(color.detach().abs().max()) == 0.0 and float(allmap.detach().abs().max()) == 0.0 and radii.numel() == 0
    (color.sum() + allmap.sum()).backward()
    assert m3.grad.shape == (0, 3)


def test_everything_behind_camera(cuda_device):
    from lara_b200 import scene as S
    sc = S.scene(1000, 0)
    cam = S.cameras(1, 64, 64, 0)[0]
    sc["means3D"] = sc["means3D"] * 0.05 + cam.c2w[:3, 3] * 1.5     # behind the camera
    out = run_candidate(sc, cam, torch.ones(3), cuda_device, grads=S.upstream_grads(64, 64, 0))
    assert out["num_rendered"] == 0 and int(out["radii"].max()) == 0
    assert np.allclose(out["color"], 1.0) and float(np.abs(out["allmap"]).max()) == 0.0
    for k in ("g_means3D", "g_sh", "g_opacities", "g_scales", "g_rotations", "g_means2D"):
        assert float(np.abs(out[k]).max()) == 0.0, k


HUGE = [(3000, 2049), (20000, 16385), (70000, 65537)]
PILEUP = [(2000, 16), (8000, 16), (8000, 48)]


def huge_splats_scene(n_big):
    from lara_b200 import scene as S
    H = W = 64
    sc = S.scene(n_big, 3)
    sc["scales"][:] = 0.6                       # every splat covers the whole image
    sc["opacities"][:] = 0.02
    sc["means3D"] *= 0.2
    sc["means3D"][::7] = sc["means3D"][0]       # exact depth ties, broken by Gaussian index
    return sc, S.cameras(1, H, W, 0)[0], torch.zeros(3)


@pytest.mark.parametrize("n_big,expect_min", HUGE)
def test_huge_splats_cover_every_tile(cuda_device, n_big, expect_min):
    """> 2048 instances per tile -> 1024-thread shared-memory bucket sort; > 8192 -> in-place global
    bitonic sort; > 65536 instances in one tile is the SURVEY's stress case."""
    from lara_b200 import scene as S
    sc, cam, bg = huge_splats_scene(n_big)
    mine = run_candidate(sc, cam, bg, cuda_device, grads=S.upstream_grads(64, 64, 1))
    counts = mine["ranges"][:, 1] - mine["ranges"][:, 0]
    assert int(counts.max()) >= expect_min
    r = Reference(f"huge_splats-{n_big}")
    assert mine["num_rendered"] == r["num_rendered"]
    assert r.equal("point_list", mine["point_list"])
    assert r.equal("ranges", mine["ranges"])
    assert r.equal("n_contrib", mine["n_contrib"][0])
    assert r.equal("allmap", mine["allmap"])
    for k in ("g_means3D", "g_opacities", "g_scales"):
        assert np.isfinite(mine[k]).all()


def pileup_scene(n, H):
    from lara_b200 import scene as S
    sc = S.scene(n, 9)
    sc["means3D"][:] = torch.tensor([0.0, 0.0, 0.0])      # all splats at the origin: identical view-space depth
    sc["scales"][:] = 0.5
    sc["opacities"][:] = 0.01
    return sc, S.cameras(1, H, H, 0)[0], torch.zeros(3)


@pytest.mark.parametrize("n,H", PILEUP)
def test_equal_depth_pileup_is_sorted_and_not_quadratic(cuda_device, n, H):
    """Every instance of a tile has the SAME depth (the degenerate case of the depth-bucket sort: one bucket holds the
    whole tile, ranking inside it would be quadratic -- 8192 instances = 65k steps per thread).  The sort falls back to the
    comparison network; order (by Gaussian index, as the reference's stable sort leaves it) and a time bound are checked."""
    from lara_b200 import rasterizer as R, scene as S
    sc, cam, bg = pileup_scene(n, H)
    mine = run_candidate(sc, cam, bg, cuda_device)
    scd = to_dev(sc, cuda_device)
    r = Reference(f"pileup-{n}_{H}")
    assert mine["num_rendered"] == r["num_rendered"] >= n
    assert r.equal("point_list", mine["point_list"])
    assert len(np.unique(mine["depths"][mine["radii"] > 0].view(np.int32))) == 1
    # time: the whole forward of this tiny image, repeated; a quadratic rank loop takes milliseconds per tile
    stm = S.settings_for(cam, bg, 1, cuda_device, R.GaussianRasterizationSettings)
    args = (scd["means3D"], scd["shs"], None, scd["opacities"], scd["scales"], scd["rotations"], None, stm)
    for _ in range(3):
        R.forward_raw(*args)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        R.forward_raw(*args)
    e1.record()
    torch.cuda.synchronize()
    assert e0.elapsed_time(e1) / 10 < 3.0, f"{e0.elapsed_time(e1) / 10:.2f} ms per forward"


def test_sorted_by_depth_then_index_within_each_tile(cuda_device):
    from lara_b200 import scene as S
    sc = S.scene(30000, 5)
    sc["means3D"][1000:2000] = sc["means3D"][0:1000]     # duplicates -> tied depths
    cam = S.cameras(1, 256, 256, 0)[0]
    out = run_candidate(sc, cam, torch.ones(3), cuda_device)
    depth_bits = out["depths"].view(np.uint32).astype(np.uint64)
    pl = out["point_list"].astype(np.int64)
    key = (depth_bits[pl] << np.uint64(32)) | pl.astype(np.uint64)
    total = 0
    for s, e in out["ranges"]:
        if e > s:
            assert np.all(np.diff(key[s:e].astype(np.float64)) >= 0) and np.all(key[s + 1:e] > key[s:e - 1])
            total += e - s
    assert total == out["num_rendered"] == int(out["tiles_touched"].sum())


def opacity_extremes_scene():
    from lara_b200 import scene as S
    sc = S.scene(8000, 6)
    sc["opacities"][0::3] = 1.0        # alpha clamps at 0.99, pixels saturate (early termination)
    sc["opacities"][1::3] = 1e-5       # never reaches 1/255
    sc["scales"] *= 3.0
    return sc, S.cameras(1, 128, 128, 0)[0], torch.full((3,), 0.5)


def test_opacity_extremes_and_saturation(cuda_device):
    from lara_b200 import scene as S
    sc, cam, bg = opacity_extremes_scene()
    gc, ga = S.upstream_grads(128, 128, 2)
    mine = run_candidate(sc, cam, bg, cuda_device, grads=(gc, ga))
    r = Reference("opacity_extremes")
    assert r.equal("n_contrib", mine["n_contrib"][0])
    assert r.equal("allmap", mine["allmap"])
    assert float(mine["accum"][0].min()) < 1e-3           # saturated pixels exist
    assert float(np.abs(mine["g_opacities"][1::3]).max()) == 0.0
    for k in ("g_means3D", "g_sh", "g_opacities", "g_scales", "g_rotations"):
        assert np.isfinite(mine[k]).all(), k


def test_capacity_overflow_reruns_binning(cuda_device, monkeypatch):
    from lara_b200 import rasterizer as R
    from lara_b200 import scene as S
    sc = S.scene(20000, 7)
    cam = S.cameras(1, 256, 256, 0)[0]
    base = run_candidate(sc, cam, torch.ones(3), cuda_device)
    monkeypatch.setattr(R, "initial_capacity", lambda P, device: 1000)   # far too small -> overflow path
    small = run_candidate(sc, cam, torch.ones(3), cuda_device)
    assert small["num_rendered"] == base["num_rendered"] > 1000
    assert np.array_equal(small["point_list"], base["point_list"])
    assert np.array_equal(small["color"].view(np.int32), base["color"].view(np.int32))
    assert np.array_equal(small["allmap"].view(np.int32), base["allmap"].view(np.int32))


def colors_precomp_outputs(mod, dev):
    """Colour and aux maps (bit for bit) and the gradients of colors_precomp and means3D through package `mod`."""
    from lara_b200 import scene as S
    sc = S.scene(5000, 8)
    cam = S.cameras(1, 128, 128, 0)[0]
    scd = to_dev(sc, dev)
    colors = torch.rand((5000, 3), generator=torch.Generator().manual_seed(8)).to(dev)
    gc, ga = [t.to(dev) for t in S.upstream_grads(128, 128, 0)]
    st = S.settings_for(cam, torch.ones(3), 1, dev, mod.GaussianRasterizationSettings)
    c_in = colors.clone().requires_grad_(True)
    m3 = scd["means3D"].clone().requires_grad_(True)
    c, rd, am = mod.GaussianRasterizer(raster_settings=st)(
        means3D=m3, means2D=torch.zeros_like(m3), colors_precomp=c_in, opacities=scd["opacities"],
        scales=scd["scales"], rotations=scd["rotations"])
    torch.autograd.backward((c, am), (gc, ga))
    return {"exact": {"color": c.detach().cpu().numpy(), "allmap": am.detach().cpu().numpy()},
            "close": {"g_colors": c_in.grad.cpu().numpy(), "g_means3D": m3.grad.cpu().numpy()}}


def test_colors_precomp_path(cuda_device):
    import diff_surfel_rasterization as DSR
    mine = colors_precomp_outputs(DSR, cuda_device)
    r = Reference("colors_precomp")
    assert r.equal("color", mine["exact"]["color"])     # no SH -> colour bit-exact too
    assert r.equal("allmap", mine["exact"]["allmap"])
    for k, v in mine["close"].items():
        assert r.rel_err(k, v) < 1e-4, k


def mark_visible_scene():
    from lara_b200 import scene as S
    sc = S.scene(10000, 9)
    sc["means3D"] = sc["means3D"] * 4.0          # some points end up behind the near plane
    return sc, S.cameras(1, 64, 64, 0)[0]


def test_mark_visible_matches_reference(cuda_device):
    from lara_b200 import scene as S
    import diff_surfel_rasterization as DSR
    sc, cam = mark_visible_scene()
    st = S.settings_for(cam, torch.ones(3), 1, cuda_device, DSR.GaussianRasterizationSettings)
    vis = DSR.GaussianRasterizer(raster_settings=st).markVisible(sc["means3D"].to(cuda_device)).cpu().numpy()
    assert vis.dtype == np.bool_ and Reference("mark_visible").equal("visible", vis) and 0 < vis.sum() < 10000


def test_non_contiguous_inputs_and_debug_flag(cuda_device):
    from lara_b200 import scene as S
    import diff_surfel_rasterization as DSR
    sc = S.scene(3000, 10)
    cam = S.cameras(1, 64, 64, 0)[0]
    scd = to_dev(sc, cuda_device)
    st = S.settings_for(cam, torch.ones(3), 1, cuda_device, DSR.GaussianRasterizationSettings, debug=True)
    rast = DSR.GaussianRasterizer(raster_settings=st)
    wide = torch.zeros(3000, 6, device=cuda_device)
    wide[:, ::2] = scd["means3D"]
    a = rast(means3D=wide[:, ::2], means2D=torch.zeros(3000, 3, device=cuda_device), shs=scd["shs"],
             opacities=scd["opacities"], scales=scd["scales"], rotations=scd["rotations"])
    b = rast(means3D=scd["means3D"], means2D=torch.zeros(3000, 3, device=cuda_device), shs=scd["shs"],
             opacities=scd["opacities"], scales=scd["scales"], rotations=scd["rotations"])
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) and torch.equal(a[1], b[1])
    with pytest.raises(RuntimeError, match="Float"):
        rast(means3D=scd["means3D"].double(), means2D=torch.zeros(3000, 3, device=cuda_device), shs=scd["shs"],
             opacities=scd["opacities"], scales=scd["scales"], rotations=scd["rotations"])


def test_outputs_can_be_modified_in_place_and_settings_may_be_strided(cuda_device):
    """Callers clamp / scale the returned images in place; MiniCam passes a transposed (strided)
    view matrix.  Both must work and give the same result as the plain call."""
    from lara_b200 import scene as S
    import diff_surfel_rasterization as DSR
    sc = S.scene(3000, 12)
    cam = S.cameras(1, 64, 64, 0)[0]
    scd = to_dev(sc, cuda_device)
    st = S.settings_for(cam, torch.ones(3), 1, cuda_device, DSR.GaussianRasterizationSettings)
    st_strided = st._replace(viewmatrix=st.viewmatrix.t().contiguous().t())
    assert not st_strided.viewmatrix.is_contiguous()
    outs = []
    for s_ in (st, st_strided):
        m3 = scd["means3D"].clone().requires_grad_(True)
        img, radii, allmap = DSR.GaussianRasterizer(raster_settings=s_)(
            means3D=m3, means2D=torch.zeros_like(m3), shs=scd["shs"], opacities=scd["opacities"],
            scales=scd["scales"], rotations=scd["rotations"])
        ref_img = img.detach().clone()
        img = img * 1.0
        img.clamp_(0.0, 0.5)            # in place on a function of the output
        allmap2 = allmap.detach().clone()
        (img.sum() + allmap.sum()).backward()
        assert torch.isfinite(m3.grad).all()
        outs.append((ref_img, allmap2, m3.grad.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert torch.allclose(outs[0][2], outs[1][2], rtol=1e-4, atol=1e-8)
