"""Fused render_img epilogue (next-row, SURVEY 8f rank 2) against the torch ops it replaces.

* CPU: the torch restatement in lara_b200/epilogue.py is pinned bit for bit against what the reference's own
  Renderer.render_img (lightning/renderer_2dgs.py) computes on the CPU with a stand-in rasterizer that returns
  fixed tensors -- the epilogue there is pure torch (tests/golden/reference, made by
  tests/golden/make_reference_golden.py).
* GPU: the fused kernel vs the restatement, forward and backward (autograd), tolerance 1e-5 of the
  tensor maximum; gradients compared where alpha > 0 (the reference's D/alpha backward is NaN at
  alpha == 0, the fused one is 0)."""
import types

import numpy as np
import pytest
import torch

from helpers import Reference, rel_err

DEPTH_RATIOS = (0.0, 0.3)


def _inputs(H, W, seed, dev="cpu"):
    g = torch.Generator().manual_seed(seed)
    color = torch.rand((3, H, W), generator=g) * 1.4 - 0.2               # exercises both clamp sides
    allmap = torch.rand((8, H, W), generator=g)
    allmap[0] = allmap[0] * 2.0 + 0.5                                    # accumulated depth
    allmap[1] = allmap[1].clamp(0.05, 1.0)
    allmap[1, : H // 4] = 0.0                                            # empty rows: alpha == 0 -> nan_to_num path
    allmap[0, : H // 4] = 0.0
    allmap[2:5] = allmap[2:5] - 0.5
    allmap[5] = allmap[5] * 2.0 + 0.5
    rays = torch.cat([torch.randn((H, W, 3), generator=g) * 0.01 + torch.tensor([0.0, 0.0, -1.9]),
                      torch.nn.functional.normalize(torch.randn((H, W, 3), generator=g) * 0.2 + torch.tensor([0.0, 0.0, 1.0]), dim=-1)], dim=-1)
    q, _ = torch.linalg.qr(torch.randn((3, 3), generator=g))
    vm = torch.eye(4); vm[:3, :3] = q; vm[3, :3] = torch.randn(3, generator=g)
    return [t.to(dev) for t in (color, allmap, rays, vm)]


@pytest.mark.parametrize("depth_ratio", DEPTH_RATIOS)
def test_torch_restatement_matches_reference_renderer_on_cpu(depth_ratio):
    from oracle.torch_restatements import render_img_epilogue_torch
    color, allmap, rays, vm = _inputs(24, 40, 0)
    mine = render_img_epilogue_torch(color, allmap, rays, vm, depth_ratio)
    ref = Reference(f"epilogue_torch-{depth_ratio}")
    assert ",".join(sorted(mine)) == ref["keys"]
    for k in mine:
        assert ref.equal(k, mine[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,depth_ratio", [(64, 64, 0.0), (50, 72, 0.3), (512, 512, 0.0)])
def test_fused_epilogue_matches_torch_ops(cuda_device, H, W, depth_ratio):
    from lara_b200.epilogue import render_img_epilogue
    from oracle.torch_restatements import render_img_epilogue_torch
    color, allmap, rays, vm = _inputs(H, W, 1, cuda_device)
    g = torch.Generator().manual_seed(5)
    weights = {"image": torch.randn((H, W, 3), generator=g), "depth": torch.randn((H, W, 1), generator=g),
               "acc_map": torch.randn((H, W), generator=g), "rend_normal": torch.randn((H, W, 3), generator=g),
               "depth_normal": torch.randn((H, W, 3), generator=g), "rend_dist": torch.randn((H, W), generator=g)}
    weights = {k: v.to(cuda_device) for k, v in weights.items()}
    res = []
    for fn in (render_img_epilogue, render_img_epilogue_torch):
        c = color.clone().requires_grad_(True)
        a = allmap.clone().requires_grad_(True)
        out = fn(c, a, rays, vm, depth_ratio)
        loss = sum((out[k] * weights[k]).sum() for k in weights)
        loss.backward()
        res.append(({k: v.detach().cpu().numpy() for k, v in out.items()}, c.grad.cpu().numpy(), a.grad.cpu().numpy()))
    (o1, dc1, da1), (o2, dc2, da2) = res
    for k in o2:
        assert o1[k].shape == o2[k].shape, k
        # the pseudo normals are a normalised cross product of differences of nearby points: a few
        # ulps of cancellation error, so 1e-4 there, 1e-5 for the element-wise outputs
        assert rel_err(o1[k], o2[k]) < (1e-4 if k == "depth_normal" else 1e-5), k
    assert rel_err(dc1, dc2) < 1e-5
    ok = (allmap[1] > 0).cpu().numpy()
    assert np.isfinite(da1).all()                       # no NaN from 0/0, unlike the torch graph
    assert not np.isfinite(da2[0][~ok]).all()           # ... which does produce them at alpha == 0
    for ch in range(8):
        assert rel_err(da1[ch][ok], da2[ch][ok]) < 1e-4, ch
    assert float(np.abs(da1[7]).max()) == 0.0


@pytest.mark.gpu
def test_fused_epilogue_feeds_rasterizer_backward(cuda_device):
    """End to end: rasterizer -> fused epilogue -> loss -> gradients of the Gaussian parameters equal
    those of rasterizer -> torch epilogue."""
    import diff_surfel_rasterization as DSR
    from lara_b200 import scene as S
    from lara_b200.epilogue import render_img_epilogue
    from oracle.torch_restatements import render_img_epilogue_torch
    dev = cuda_device
    sc = S.scene(20000, 4)
    cam = S.cameras(1, 128, 128, 0)[0]
    st = S.settings_for(cam, torch.ones(3), 1, dev, DSR.GaussianRasterizationSettings)
    _, _, rays, _ = _inputs(128, 128, 2, dev)
    grads = []
    for fn in (render_img_epilogue, render_img_epilogue_torch):
        leaves = {k: sc[k].to(dev).requires_grad_(True) for k in ("means3D", "shs", "opacities", "scales", "rotations")}
        img, radii, allmap = DSR.GaussianRasterizer(raster_settings=st)(
            means3D=leaves["means3D"], means2D=torch.zeros_like(leaves["means3D"]), shs=leaves["shs"],
            opacities=leaves["opacities"], scales=leaves["scales"], rotations=leaves["rotations"])
        out = fn(img, allmap + 0.0, rays, st.viewmatrix, 0.0)
        mask = (allmap[1] > 0).detach()
        loss = ((out["image"] - 0.4) ** 2).mean() + 0.2 * (out["rend_normal"] ** 2).mean() + out["rend_dist"].mean() \
            + 0.1 * (out["depth"][..., 0] * mask).mean() + out["acc_map"].mean() + 0.05 * (out["depth_normal"] * out["rend_normal"].detach()).sum(-1).mean()
        loss.backward()
        grads.append({k: torch.nan_to_num(v.grad).cpu().numpy() for k, v in leaves.items()})
    for k in grads[0]:
        assert rel_err(grads[0][k], grads[1][k]) < 1e-4, k


@pytest.mark.gpu
@pytest.mark.parametrize("sh_degree", [0, 1])
def test_fused_activations_match_torch_activations(cuda_device, sh_degree):
    """raw_activations=True (sigmoid / exp / normalize inside the kernels) against the same
    rasterizer fed with torch's activations: forward bit-identical, raw-parameter gradients 1e-5."""
    import diff_surfel_rasterization as DSR
    from lara_b200 import scene as S
    dev = cuda_device
    sc = S.scene(40000, 9, sh_degree=sh_degree)
    cam = S.cameras(1, 160, 192, 2)[0]
    st = S.settings_for(cam, torch.ones(3), sh_degree, dev, DSR.GaussianRasterizationSettings)
    base = {"means3D": sc["means3D"], "shs": sc["shs"], "opacities": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
            "scales": torch.log(sc["scales"]), "rotations": sc["rotations"] * 1.7}
    g = torch.Generator().manual_seed(3)
    w_img = torch.randn((3, 160, 192), generator=g).to(dev)
    w_all = torch.randn((8, 160, 192), generator=g).to(dev)
    res = []
    for raw in (True, False):
        leaves = {k: v.to(dev).clone().requires_grad_(True) for k, v in base.items()}
        kw = dict(opacities=leaves["opacities"], scales=leaves["scales"], rotations=leaves["rotations"])
        if not raw:
            kw = dict(opacities=torch.sigmoid(leaves["opacities"]), scales=torch.exp(leaves["scales"]),
                      rotations=torch.nn.functional.normalize(leaves["rotations"]))
        means2D = torch.zeros_like(leaves["means3D"], requires_grad=True)
        rast = DSR.GaussianRasterizer(raster_settings=st)
        img, radii, allmap = (rast.forward_raw_activations if raw else rast)(
            means3D=leaves["means3D"], means2D=means2D, shs=leaves["shs"], **kw)
        ((img * w_img).sum() + (allmap * w_all).sum()).backward()
        res.append((img.detach().cpu().numpy(), allmap.detach().cpu().numpy(), radii.cpu().numpy(),
                    {k: v.grad.cpu().numpy() for k, v in leaves.items()}, means2D.grad.cpu().numpy()))
    a, b = res
    assert np.array_equal(a[2], b[2])
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    for k in a[3]:
        assert np.isfinite(a[3][k]).all(), k
        assert rel_err(a[3][k], b[3][k]) < 1e-5, k
    assert rel_err(a[4], b[4]) < 1e-5


def _pipeline_setup(dev):
    import types
    from lara_b200 import scene as S
    H = W = 160
    sc = S.scene(30000, 21)
    c = S.cameras(2, H, W, 5)[1]
    cam = types.SimpleNamespace(image_height=H, image_width=W, FoVx=0.75, FoVy=0.75,
                                world_view_transform=c.viewmatrix.to(dev), full_proj_transform=c.projmatrix.to(dev),
                                camera_center=c.campos.to(dev))
    _, _, rays, _ = _inputs(H, W, 3, dev)
    base = {"centers": sc["means3D"], "shs": sc["shs"], "opacity": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
            "scales": torch.log(sc["scales"]), "rotations": sc["rotations"] * 0.7}
    raw = {k: v.to(dev).clone().requires_grad_(True) for k, v in base.items()}
    return c, cam, rays, raw


def _pipeline_loss_and_outputs(out, raw):
    mask = (out["acc_map"] > 0).detach()
    loss = ((out["image"] - 0.4) ** 2).mean() + 0.2 * (out["rend_normal"] ** 2).mean() + 1000.0 * out["rend_dist"].mean() \
        + 0.1 * (out["depth"][..., 0] * mask).mean() + out["acc_map"].mean() \
        + 0.2 * (1 - (out["rend_normal"] * out["depth_normal"]).sum(-1)).mean()
    loss.backward()
    return {"close": {**{k: v.detach().cpu().numpy() for k, v in out.items()},
                      **{"grad." + k: torch.nan_to_num(v.grad).cpu().numpy() for k, v in raw.items()}},
            "scalars": {"keys": ",".join(sorted(out))}}


def reference_pipeline_outputs(mod, dev):
    """The pipeline LaRa runs today: the rasterizer of package `mod` + the torch epilogue."""
    from lara_b200 import scene as S
    from oracle.torch_restatements import render_img_epilogue_torch
    c, cam, rays, raw = _pipeline_setup(dev)
    rs = S.settings_for(c, torch.ones(3), 1, dev, mod.GaussianRasterizationSettings)
    img, radii, allmap = mod.GaussianRasterizer(raster_settings=rs)(
        means3D=raw["centers"], means2D=torch.zeros_like(raw["centers"], requires_grad=True) + 0, shs=raw["shs"],
        opacities=torch.sigmoid(raw["opacity"]), scales=torch.exp(raw["scales"]),
        rotations=torch.nn.functional.normalize(raw["rotations"]), cov3D_precomp=None)
    return _pipeline_loss_and_outputs(render_img_epilogue_torch(img, allmap, rays, cam.world_view_transform, 0.0), raw)


@pytest.mark.gpu
@pytest.mark.parametrize("fused_activations", [True, False])
def test_fast_renderer_matches_reference_pipeline(cuda_device, fused_activations):
    """lara_b200.renderer.Renderer.render_img == reference rasterizer + the torch epilogue (the
    pipeline LaRa runs today, stored by reference_pipeline_outputs), images and raw-parameter gradients."""
    from lara_b200.renderer import Renderer
    dev = cuda_device
    _, cam, rays, raw = _pipeline_setup(dev)
    r = Renderer(sh_degree=1, white_background=True, fused_activations=fused_activations)
    out = r.render_img(cam, rays, raw["centers"], raw["shs"], raw["opacity"], raw["scales"], raw["rotations"], dev)
    mine = _pipeline_loss_and_outputs(out, raw)["close"]
    ref = Reference("fast_renderer_pipeline")
    assert ",".join(sorted(out)) == ref["keys"] == "acc_map,depth,depth_normal,image,rend_dist,rend_normal"
    for k in out:
        assert ref.rel_err(k, mine[k]) < (1e-4 if k == "depth_normal" else 1e-5), k
    for k in raw:
        assert np.isfinite(mine["grad." + k]).all()
        assert ref.rel_err("grad." + k, mine["grad." + k]) < 2e-4, k


@pytest.mark.gpu
@pytest.mark.parametrize("streams,fused_activations", [(1, True), (3, True), (3, False)])
def test_render_views_matches_per_view_loop(cuda_device, streams, fused_activations):
    """Renderer.render_views (one autograd node, multi-stream, in-kernel gradient accumulation) ==
    the per-view loop of network.py:486-495 + the cat of :525: outputs bit-identical (same kernels),
    raw-parameter gradients to 1e-5 (different summation order across views)."""
    import types
    from lara_b200 import scene as S
    from lara_b200.multiview import concat_views
    from lara_b200.renderer import Renderer
    dev = cuda_device
    H = W = 128
    V = 5
    sc = S.scene(25000, 33)
    cs = S.cameras(V, H, W, 7)
    cams = [types.SimpleNamespace(image_height=H, image_width=W, FoVx=0.75, FoVy=0.75,
                                  world_view_transform=c.viewmatrix.to(dev), full_proj_transform=c.projmatrix.to(dev),
                                  camera_center=c.campos.to(dev)) for c in cs]
    rays = torch.stack([_inputs(H, W, 10 + v, dev)[2] for v in range(V)])
    bgs = torch.tensor([[1.0, 1.0, 1.0], [0.0, 0.0, 0.0], [0.5, 0.5, 0.5], [1.0, 1.0, 1.0], [0.0, 0.0, 0.0]])
    base = {"centers": sc["means3D"], "shs": sc["shs"], "opacity": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
            "scales": torch.log(sc["scales"]), "rotations": sc["rotations"] * 0.7}
    g = torch.Generator().manual_seed(11)
    tar = torch.rand((H, V * W, 3), generator=g).to(dev)

    def loss_of(out):
        return ((out["image"] - tar) ** 2).mean() + 1000.0 * out["rend_dist"].mean() \
            + 0.2 * ((1 - (out["rend_normal"] * out["depth_normal"]).sum(-1)) * out["acc_map"].detach()).mean() \
            + 0.1 * (out["depth"][..., 0] * (out["acc_map"] > 0).detach()).mean()

    r = Renderer(sh_degree=1, white_background=True, fused_activations=fused_activations)
    res = []
    for batched in (True, False):
        raw = {k: v.to(dev).clone().requires_grad_(True) for k, v in base.items()}
        if batched:
            out = concat_views(r.render_views(cams, rays, raw["centers"], raw["shs"], raw["opacity"], raw["scales"],
                                              raw["rotations"], dev, bg_colors=bgs, streams=streams))
        else:
            frames = []
            for j, cam in enumerate(cams):
                r.set_bg_color(bgs[j])
                frames.append(r.render_img(cam, rays[j], raw["centers"], raw["shs"], raw["opacity"], raw["scales"],
                                           raw["rotations"], dev))
            out = {k: torch.cat([f[k] for f in frames], dim=1) for k in frames[0]}
        loss_of(out).backward()
        res.append(({k: v.detach().cpu().numpy() for k, v in out.items()}, {k: v.grad.cpu().numpy() for k, v in raw.items()}))
    (o1, g1), (o2, g2) = res
    assert sorted(o1) == sorted(o2)
    for k in o2:
        assert o1[k].shape == o2[k].shape, k
        assert np.array_equal(o1[k].view(np.uint32), o2[k].view(np.uint32)), k
    for k in g1:
        assert np.isfinite(g1[k]).all(), k
        assert rel_err(g1[k], g2[k]) < 1e-5, k


@pytest.mark.gpu
def test_render_views_without_rays_returns_clamped_images(cuda_device):
    import types
    from lara_b200 import scene as S
    from lara_b200.renderer import Renderer
    dev = cuda_device
    H = W = 96
    sc = S.scene(8000, 2)
    cs = S.cameras(3, H, W, 1)
    cams = [types.SimpleNamespace(image_height=H, image_width=W, FoVx=0.75, FoVy=0.75,
                                  world_view_transform=c.viewmatrix.to(dev), full_proj_transform=c.projmatrix.to(dev),
                                  camera_center=c.campos.to(dev)) for c in cs]
    raw = {"centers": sc["means3D"], "shs": sc["shs"] * 3.0, "opacity": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
           "scales": torch.log(sc["scales"]), "rotations": sc["rotations"]}
    r = Renderer(sh_degree=1, white_background=False)
    res = []
    for batched in (True, False):
        leaves = {k: v.to(dev).clone().requires_grad_(True) for k, v in raw.items()}
        args = (leaves["centers"], leaves["shs"], leaves["opacity"], leaves["scales"], leaves["rotations"], dev)
        if batched:
            img = r.render_views(cams, None, *args)["image"]
        else:
            img = torch.stack([r.render_img(cam, None, *args) for cam in cams])
        (img ** 2).sum().backward()
        res.append((img.detach().cpu().numpy(), {k: v.grad.cpu().numpy() for k, v in leaves.items()}))
    assert res[0][0].shape == res[1][0].shape == (3, 3, H, W)
    assert np.array_equal(res[0][0], res[1][0])
    for k in res[0][1]:
        assert rel_err(res[0][1][k], res[1][1][k]) < 1e-5, k
