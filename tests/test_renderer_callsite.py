"""The consumer: LaRa's lightning/renderer_2dgs.py must run unchanged on top of this package.

* GPU: the call pattern of Renderer.render_img (renderer_2dgs.py:167-268) -- activations,
  zeros+0 screenspace tensor with retain_grad, keyword call, the torch post-processing of the aux
  maps and a loss -- is replayed with this package; images and the gradients wrt the *raw* network
  outputs must agree with what the reference build computes (tests/golden/reference).
"""
import numpy as np
import pytest
import torch

from helpers import Reference


def raw_parameters(sc):
    """Raw network outputs as LaRa's decoder hands them to render_img (activations still to apply)."""
    return {"centers": sc["means3D"], "shs": sc["shs"], "opacity": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
            "scales": torch.log(sc["scales"]), "rotations": sc["rotations"] * 1.7}


def _render_img_like(mod, cam, raw, bg, dev):
    """Replays renderer_2dgs.Renderer.render_img with module `mod` as the rasterizer package."""
    from lara_b200 import scene as S
    rs = S.settings_for(cam, bg, 1, dev, mod.GaussianRasterizationSettings)
    # MiniCam hands over w2c.transpose(0, 1): a NON-contiguous view matrix (lightning/utils.py:40)
    w2c = rs.viewmatrix.t().contiguous()
    rs = rs._replace(viewmatrix=w2c.transpose(0, 1))
    assert not rs.viewmatrix.is_contiguous()
    rast = mod.GaussianRasterizer(raster_settings=rs)
    opacity = torch.sigmoid(raw["opacity"])
    scales = torch.exp(raw["scales"])
    rotations = torch.nn.functional.normalize(raw["rotations"])
    centers = raw["centers"]
    screenspace = torch.zeros_like(centers, dtype=centers.dtype, requires_grad=True, device=dev) + 0
    screenspace.retain_grad()
    img, radii, allmap = rast(means3D=centers, means2D=screenspace, shs=raw["shs"], opacities=opacity,
                              scales=scales, rotations=rotations, cov3D_precomp=None)
    img = img.clamp(0, 1)
    alpha = allmap[1:2]
    normal = (allmap[2:5].permute(1, 2, 0) @ (rs.viewmatrix[:3, :3].T)).permute(2, 0, 1)
    # (LaRa divides by alpha and nan_to_num()s the result; with anomaly mode on, 0/0 at empty pixels
    #  would trip DivBackward itself, so the replay guards the denominator)
    depth = torch.nan_to_num(allmap[0:1] / alpha.clamp_min(1e-6), 0, 0)
    dist = allmap[6:7]
    loss = ((img - 0.3) ** 2).mean() + 0.2 * (normal ** 2).mean() + 1000.0 * dist.mean() + 0.1 * depth.mean() + alpha.mean()
    return img, allmap, radii, loss, screenspace


@pytest.mark.gpu
def test_render_img_call_pattern_matches_reference(cuda_device):
    import diff_surfel_rasterization as DSR
    from lara_b200 import scene as S
    dev = cuda_device
    sc = S.scene(20000, 11)
    cam = S.cameras(2, 160, 160, 3)[1]
    raw = {k: v.to(dev).clone().requires_grad_(True) for k, v in raw_parameters(sc).items()}
    with torch.autograd.set_detect_anomaly(True):
        img, allmap, radii, loss, ss = _render_img_like(DSR, cam, raw, torch.ones(3), dev)
        loss.backward()
    r = Reference("render_img_call_pattern")
    assert r.equal("image", img)
    assert r.equal("allmap", allmap)
    assert r.equal("radii", radii)
    assert float(loss) == r["loss"]
    for k, v in raw.items():
        g = v.grad.cpu().numpy()
        assert np.isfinite(g).all()
        assert r.rel_err("grad." + k, g) < 1e-4, k
    assert r.rel_err("grad.means2D", ss.grad) < 1e-4        # viewspace (means2D) gradient used for densification statistics
