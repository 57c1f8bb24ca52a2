"""Deferred instance-count read-back (DESIGN.md section 4): a forward returns without waiting; the count is an int-like
object resolved on demand; an overflowed optimistic capacity is repaired in place (with a warning) when the count is
resolved -- at the latest when the backward starts -- and `debug=True` restores the check inside the forward."""
import warnings

import numpy as np
import pytest
import torch

from helpers import Reference, to_dev

pytestmark = pytest.mark.gpu

KEYS = ("means3D", "shs", "opacities", "scales", "rotations")


def _leaves(scd):
    return {k: scd[k].clone().requires_grad_(True) for k in KEYS}


def _render(DSR, leaves, st):
    m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)
    rast = DSR.GaussianRasterizer(raster_settings=st)
    return rast(means3D=leaves["means3D"], means2D=m2d, shs=leaves["shs"], opacities=leaves["opacities"],
                scales=leaves["scales"], rotations=leaves["rotations"])


def test_ctx_num_rendered_is_lazy_and_correct(cuda_device):
    import diff_surfel_rasterization as DSR
    from lara_b200 import rasterizer as R, scene as S
    sc = S.scene(20000, 11)
    scd = to_dev(sc, cuda_device)
    cam = S.cameras(1, 256, 256, 1)[0]
    st = S.settings_for(cam, torch.ones(3), 1, cuda_device, DSR.GaussianRasterizationSettings)
    color, radii, allmap = _render(DSR, _leaves(scd), st)
    n = color.grad_fn.num_rendered                     # the reference stores an int on ctx (DSR __init__.py:95)
    assert isinstance(n, (int, R.LazyCount))
    assert int(n) == Reference("ctx_num_rendered")["num_rendered"]      # what the reference's forward counts
    assert n == int(n) and f"{n}" == str(int(n))


def test_overflow_is_repaired_before_the_backward_with_a_warning(cuda_device, monkeypatch):
    import diff_surfel_rasterization as DSR
    from lara_b200 import rasterizer as R, scene as S
    sc = S.scene(20000, 12)
    scd = to_dev(sc, cuda_device)
    cam = S.cameras(1, 256, 256, 2)[0]
    st = S.settings_for(cam, torch.ones(3), 1, cuda_device, DSR.GaussianRasterizationSettings)
    gc, ga = [t.to(cuda_device) for t in S.upstream_grads(256, 256, 3)]

    def run():
        lv = _leaves(scd)
        color, radii, allmap = _render(DSR, lv, st)
        torch.autograd.backward((color, allmap), (gc, ga))
        torch.cuda.synchronize()
        return color.detach().clone(), {k: v.grad.clone() for k, v in lv.items()}
    c0, g0 = run()
    monkeypatch.setattr(R, "initial_capacity", lambda P, device: 1000)       # far too small: every tile list overflows
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        c1, g1 = run()
    assert any(issubclass(x.category, RuntimeWarning) and "optimistic capacity" in str(x.message) for x in w)
    assert torch.equal(c0, c1)                                               # the image was recomputed in place
    for k in g0:
        assert float((g0[k] - g1[k]).abs().max()) <= 1e-5 * float(g0[k].abs().max()), k
    # debug=True (the reference's synchronise-and-check switch): checked inside the forward, silently
    st_dbg = st._replace(debug=True)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        color, radii, allmap = _render(DSR, _leaves(scd), st_dbg)
    assert not [x for x in w if issubclass(x.category, RuntimeWarning)]
    assert torch.equal(color.detach(), c0)


def test_batched_views_overflow_is_repaired(cuda_device, monkeypatch):
    from lara_b200 import rasterizer as R, scene as S
    sc = S.scene(15000, 13)
    scd = to_dev(sc, cuda_device)
    V, H, W = 3, 128, 128
    sets = [S.settings_for(c, torch.ones(3), 1, cuda_device, R.GaussianRasterizationSettings) for c in S.cameras(V, H, W, 4)]
    cams = R.pack_cameras(sets, cuda_device)
    args = (scd["means3D"], scd["shs"], None, scd["opacities"], scd["scales"], scd["rotations"], None, cams,
            sets[0].tanfovx, sets[0].tanfovy, H, W, 1)
    c0, a0, r0, s0 = R.forward_views_raw(*args)
    counts0 = s0.num_rendered
    monkeypatch.setattr(R, "initial_capacity", lambda P, device: 512)
    with warnings.catch_warnings(record=True):
        warnings.simplefilter("always")
        c1, a1, r1, s1 = R.forward_views_raw(*args)
        counts1 = s1.num_rendered                                             # resolving repairs the overflow
    torch.cuda.synchronize()
    assert counts0 == counts1 and min(counts0) > 512 and s1.capacity >= max(counts1)
    assert torch.equal(c0, c1) and torch.equal(a0, a1)
