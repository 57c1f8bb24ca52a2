"""Fused loss -> dL/d(render_img outputs) producer (next-row, SURVEY 8f rank 3).

* CPU: the torch restatement (oracle/torch_restatements.lara_loss_torch) is pinned bit-exactly against what the
  reference's own ``Losses.forward`` (lightning/loss.py) computes with ``pytorch_msssim`` replaced by a stub whose
  MS_SSIM returns 1 -- the MSE / distortion / normal-consistency terms and their autograd gradients are the
  reference's (tests/golden/reference, made by tests/golden/make_reference_golden.py).
* GPU: ``lara_b200.loss.scene_loss`` (two CUDA kernels on the stacked planar buffers) vs the restatement on the
  concatenated [H, V*W, C] layout, loss terms and all four gradient maps, and end to end through
  ``render_scene_views`` to the Gaussian-parameter gradients."""
import types

import pytest
import torch

from helpers import Reference, rel_err

ITERATIONS = (10, 5000)


def _fake_outputs(B, V, H, W, seed, dev="cpu"):
    g = torch.Generator().manual_seed(seed)

    def r(*s):
        return torch.rand(s, generator=g)
    out = {"image": r(B, H, V * W, 3), "rend_dist": r(B, H, V * W) * 0.01, "acc_map": r(B, H, V * W),
           "rend_normal": torch.nn.functional.normalize(r(B, H, V * W, 3) - 0.5, dim=-1),
           "depth_normal": torch.nn.functional.normalize(r(B, H, V * W, 3) - 0.5, dim=-1)}
    tar = r(B, V, H, W, 3)
    return {k: v.to(dev) for k, v in out.items()}, tar.to(dev)


@pytest.mark.parametrize("it", ITERATIONS)
def test_loss_restatement_matches_reference_losses_on_cpu(it):
    from oracle.torch_restatements import lara_loss_torch
    out, tar = _fake_outputs(2, 3, 16, 24, 0)
    lb = {k: v.clone().requires_grad_(k != "acc_map") for k, v in out.items()}
    my_loss, my_stats = lara_loss_torch(lb, tar, it)
    ref = Reference(f"loss-{it}")
    assert ref.equal("loss", my_loss.reshape(()))
    for k in my_stats:
        assert ref.equal("stat." + k, my_stats[k].reshape(-1)), k
    my_loss.backward()
    assert ",".join(sorted(k for k, v in lb.items() if v.grad is None)) == ref["no_grad"]
    for k in lb:
        if lb[k].grad is not None:
            assert ref.equal("grad." + k, lb[k].grad), k


@pytest.mark.gpu
@pytest.mark.parametrize("V,H,W,it,B", [(3, 32, 48, 5000, 1), (8, 128, 128, 5000, 4), (2, 50, 72, 10, 1)])
def test_fused_scene_loss_matches_restatement(cuda_device, V, H, W, it, B):
    from lara_b200.loss import scene_loss
    from lara_b200.multiview import concat_views
    from oracle.torch_restatements import lara_loss_torch
    dev = cuda_device
    g = torch.Generator().manual_seed(V * 100 + H)
    planar = {"image": torch.rand((V, 3, H, W), generator=g), "rend_normal": torch.rand((V, 3, H, W), generator=g) - 0.5,
              "depth_normal": torch.rand((V, 3, H, W), generator=g) - 0.5, "depth": torch.rand((V, 1, H, W), generator=g)}
    flat = {"acc_map": torch.rand((V, H, W), generator=g), "rend_dist": torch.rand((V, H, W), generator=g) * 0.01}
    tar = torch.rand((V, H, W, 3), generator=g).to(dev)

    def leaves():
        d = {k: v.to(dev).clone().requires_grad_(True) for k, v in planar.items()}
        d.update({k: v.to(dev).clone().requires_grad_(True) for k, v in flat.items()})
        return d
    a, b = leaves(), leaves()
    # the stacked dict render_scene_views returns: channel-last views of planar buffers
    out_a = {k: (a[k].permute(0, 2, 3, 1) if a[k].ndim == 4 else a[k]) for k in a}
    loss_a, stats_a = scene_loss(out_a, tar, it, batch_scenes=B)
    (loss_a * 3.0).backward()                      # a non-unit upstream gradient travels through device memory
    # the reference layout: views side by side, one scene of a batch of B (means over B scenes -> scale 1/B)
    out_b = {k: v.unsqueeze(0) for k, v in concat_views({k: (b[k].permute(0, 2, 3, 1) if b[k].ndim == 4 else b[k]) for k in b}).items()}
    loss_b, stats_b = lara_loss_torch(out_b, tar.unsqueeze(0), it)
    # with B scenes every mean's denominator grows by B: emulate by scaling this scene's share
    share = 1.0 / B
    (loss_b * 3.0 * share).backward()
    assert abs(float(loss_a) - float(loss_b) * share) < 2e-6 * max(1.0, abs(float(loss_b)))
    for k in ("mse", "distortion", "normal"):
        if k in stats_b:
            assert abs(float(stats_a[k]) - float(stats_b[k]) * share) < 2e-6 * max(1.0, abs(float(stats_b[k]))), k
    for k in ("image", "rend_normal", "depth_normal", "rend_dist"):
        if b[k].grad is None:
            assert a[k].grad is None or float(a[k].grad.abs().max()) == 0.0, k
        else:
            assert rel_err(a[k].grad.cpu().numpy(), b[k].grad.cpu().numpy()) < 1e-5, k
    assert a["acc_map"].grad is None and a["depth"].grad is None       # acc_map is detached in the reference; depth unused


@pytest.mark.gpu
def test_scene_loss_end_to_end_parameter_gradients(cuda_device):
    """render_scene_views -> scene_loss -> backward == render_scene_views -> concat -> torch loss -> backward."""
    import math
    from lara_b200 import scene as S
    from lara_b200.loss import scene_loss
    from lara_b200.multiview import concat_views
    from lara_b200.renderer import Renderer
    from oracle.torch_restatements import lara_loss_torch
    dev = cuda_device
    P, H, W, V = 20000, 128, 128, 4
    sc = S.scene(P, 2)
    cams_ = S.cameras(V, H, W, 2)
    fov = 2 * math.atan(cams_[0].tanfovx)
    cams = [types.SimpleNamespace(image_height=H, image_width=W, FoVx=fov, FoVy=fov,
                                  world_view_transform=c.viewmatrix.to(dev), full_proj_transform=c.projmatrix.to(dev),
                                  camera_center=c.campos.to(dev)) for c in cams_]
    g = torch.Generator().manual_seed(5)
    rays = torch.cat([torch.zeros(V, H, W, 3), torch.nn.functional.normalize(torch.randn((V, H, W, 3), generator=g), dim=-1)], -1).to(dev)
    tar = torch.rand((V, H, W, 3), generator=g).to(dev)
    raw = {"centers": sc["means3D"], "shs": sc["shs"], "opacity": torch.logit(sc["opacities"].clamp(1e-4, 1 - 1e-4)),
           "scales": torch.log(sc["scales"]), "rotations": sc["rotations"] * 1.7}
    r = Renderer(sh_degree=1)
    grads = []
    for fused in (True, False):
        leaves = {k: v.to(dev).clone().requires_grad_(True) for k, v in raw.items()}
        out = r.render_views(cams, rays, leaves["centers"], leaves["shs"], leaves["opacity"], leaves["scales"],
                             leaves["rotations"], dev)
        if fused:
            loss, _ = scene_loss(out, tar, 5000)
        else:
            loss, _ = lara_loss_torch({k: v.unsqueeze(0) for k, v in concat_views(out).items()}, tar.unsqueeze(0), 5000)
        loss.backward()
        grads.append({k: v.grad.detach().cpu().numpy() for k, v in leaves.items()})
    for k in grads[0]:
        assert rel_err(grads[0][k], grads[1][k]) < 2e-5, k
