"""Generate tests/golden/reference/*.npz: what the UNMODIFIED reference computes for the tests that compare
this project with it, so that those tests run anywhere without the reference.

    python tests/golden/make_reference_golden.py cpu OUT_DIR    # the reference's Python modules on the CPU
    python tests/golden/make_reference_golden.py gpu OUT_DIR    # the reference rasterizer (oracle/_ref) on a B200

``cpu`` needs the reference's sources (``LARA_REFERENCE_ROOT``, as for oracle/build_ref.py), ``gpu`` needs the
oracle/_ref build.  Every case below repeats, input for input, the reference side of the test named beside it;
what is stored (tests/helpers.py save_reference) is a fingerprint of each array the test compares bit for bit,
and a seeded sample of each array it compares within a tolerance.  Copy OUT_DIR/*.npz to tests/golden/reference/.
"""
from __future__ import annotations

import functools
import importlib.util
import os
import sys
import types

import numpy as np
import torch

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)

from helpers import save_reference, tile_pixel_mask, to_dev  # noqa: E402
from lara_b200 import scene as S  # noqa: E402
from oracle.build_ref import REF_ROOT  # noqa: E402

GRAD_KEYS = ("means3D", "shs", "opacities", "scales", "rotations")


def _np(d):
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in d.items()}


def _grads(ref, scd, st, gc, ga):
    leaves = {k: scd[k].clone().requires_grad_(True) for k in GRAD_KEYS}
    m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)
    c, _, am = ref.GaussianRasterizer(raster_settings=st)(
        means3D=leaves["means3D"], means2D=m2d, shs=leaves["shs"], opacities=leaves["opacities"],
        scales=leaves["scales"], rotations=leaves["rotations"])
    torch.autograd.backward((c, am), (gc, ga))
    g = {k: v.grad.cpu().numpy() for k, v in leaves.items()}
    g["means2D"] = m2d.grad.cpu().numpy()
    return g


def _noise(g1, g2):
    from helpers import rel_err
    return {"noise." + k: rel_err(g2[k], g1[k]) for k in g1}


def _state(r, H, W):
    """The reference's forward state as test_gpu_parity / test_gpu_headline compare it."""
    vis = r["radii"] > 0
    mask = tile_pixel_mask(r["ranges"], H, W)
    return {"radii": r["radii"], "tiles_touched": r["tiles_touched"], "point_list": r["point_list"],
            "ranges": r["ranges"], "depths_vis": r["depths"][vis], "transMat_vis": r["transMat"][vis],
            "means2D_vis": r["means2D"][vis], "rgb_vis": r["rgb"][vis], "n_contrib": r["n_contrib"][0],
            "median_contributor": r["n_contrib"][1][mask], "accum": r["accum"], "allmap": r["allmap"],
            "color": r["color"]}


def gpu(out):
    from oracle import ref as REF
    import test_epilogue as TE
    import test_gpu_headline as TH
    import test_gpu_parity as TP
    import test_renderer_callsite as TR
    save = functools.partial(save_reference, out_dir=out)
    ref = REF.load()
    dev = torch.device("cuda:0")

    def forward(sc, cam, bg, deg):
        scd = to_dev(sc, dev)
        st = S.settings_for(cam, bg, deg, dev, ref.GaussianRasterizationSettings)
        return scd, st, _np(REF.forward_raw(ref, scd, st))

    # test_gpu_parity
    for P, H, W, seed, deg, bgv in TP.CASES:
        sc = S.scene(P, seed, sh_degree=deg)
        cam = S.cameras(3, H, W, seed)[seed % 3]
        scd, st, r = forward(sc, cam, torch.full((3,), bgv), deg)
        save(TP.case_name("state", P, H, W, seed), exact=_state(r, H, W), scalars={"num_rendered": r["num_rendered"]})
        if (P, H, W, seed, deg, bgv) in TP.CASES[:4]:
            gc, ga = [t.to(dev) for t in S.upstream_grads(H, W, seed)]
            g1, g2 = _grads(ref, scd, st, gc, ga), _grads(ref, scd, st, gc, ga)
            save(TP.case_name("grads", P, H, W, seed), close=g1, scalars=_noise(g1, g2))

    # test_gpu_headline
    def state_and_grads(sc, cam, bg, deg, H, W, seed, twice, prefix=""):
        scd, st, r = forward(sc, cam, bg, deg)
        gc, ga = [t.to(dev) for t in S.upstream_grads(H, W, seed)]
        g1 = _grads(ref, scd, st, gc, ga)
        g1.pop("means2D")
        scalars = {"num_rendered": r["num_rendered"]}
        if twice:
            scalars.update(_noise(g1, {k: v for k, v in _grads(ref, scd, st, gc, ga).items() if k != "means2D"}))
        p = lambda d: {prefix + k: v for k, v in d.items()}    # noqa: E731
        return p(_state(r, H, W)), p(g1), p(scalars)

    for P, size, seed in TH.HEADLINE:
        sc = S.scene(P, seed, sh_degree=1)
        cam = S.cameras(3, size, size, seed)[seed % 3]
        e, c, s = state_and_grads(sc, cam, torch.ones(3), 1, size, size, seed, True)
        save(f"headline-{P}_{size}_s{seed}", exact=e, close=c, scalars=s)
        torch.cuda.empty_cache()
    rng = np.random.default_rng(TH.SWEEP_SEED)
    exact, close, scalars = {}, {}, {}
    for it in range(25):
        tag, sc, cam = TH._sweep_config(rng)
        e, c, s = state_and_grads(sc, cam, torch.full((3,), tag["bg"]), tag["deg"], tag["H"], tag["W"], tag["seed"],
                                  False, prefix=f"{it}/")
        exact.update(e); close.update(c); scalars.update(s)
    save("sweep25", exact=exact, close=close, scalars=scalars, k=64)

    # test_gpu_edges
    import test_gpu_edges as TG
    for n_big, _ in TG.HUGE:
        sc, cam, bg = TG.huge_splats_scene(n_big)
        _, _, r = forward(sc, cam, bg, 1)
        save(f"huge_splats-{n_big}", scalars={"num_rendered": r["num_rendered"]},
             exact={"point_list": r["point_list"], "ranges": r["ranges"], "n_contrib": r["n_contrib"][0],
                    "allmap": r["allmap"]})
    for n, H in TG.PILEUP:
        sc, cam, bg = TG.pileup_scene(n, H)
        _, _, r = forward(sc, cam, bg, 1)
        save(f"pileup-{n}_{H}", scalars={"num_rendered": r["num_rendered"]}, exact={"point_list": r["point_list"]})
    sc, cam, bg = TG.opacity_extremes_scene()
    _, _, r = forward(sc, cam, bg, 1)
    save("opacity_extremes", exact={"n_contrib": r["n_contrib"][0], "allmap": r["allmap"]})
    save("colors_precomp", **TG.colors_precomp_outputs(ref, dev))
    sc, cam = TG.mark_visible_scene()
    st = S.settings_for(cam, torch.ones(3), 1, dev, ref.GaussianRasterizationSettings)
    save("mark_visible", exact={"visible": ref.GaussianRasterizer(raster_settings=st).markVisible(
        sc["means3D"].to(dev)).cpu().numpy()})

    # test_gpu_readback
    sc = S.scene(20000, 11)
    _, _, r = forward(sc, S.cameras(1, 256, 256, 1)[0], torch.ones(3), 1)
    save("ctx_num_rendered", scalars={"num_rendered": r["num_rendered"]})

    # test_epilogue: reference rasterizer + the torch epilogue
    save("fast_renderer_pipeline", **TE.reference_pipeline_outputs(ref, dev))

    # test_renderer_callsite
    sc = S.scene(20000, 11)
    cam = S.cameras(2, 160, 160, 3)[1]
    raw = {k: v.to(dev).clone().requires_grad_(True) for k, v in TR.raw_parameters(sc).items()}
    with torch.autograd.set_detect_anomaly(True):
        img, allmap, radii, loss, ss = TR._render_img_like(ref, cam, raw, torch.ones(3), dev)
        loss.backward()
    save("render_img_call_pattern", exact={"image": img, "allmap": allmap, "radii": radii},
         close={**{"grad." + k: v.grad for k, v in raw.items()}, "grad.means2D": ss.grad},
         scalars={"loss": loss.item()})


def _module(path, name, stubs=None):
    saved = {k: sys.modules.get(k) for k in (stubs or {})}
    sys.modules.update(stubs or {})
    try:
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


def _reference_network():
    """lightning/network.py with stand-ins for the packages it imports at module level but this test does not use."""
    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m
    tv = stub("torchvision")
    tv.transforms = stub("torchvision.transforms")
    stubs = {"timm": stub("timm"), "pytorch_lightning": stub("pytorch_lightning", LightningModule=torch.nn.Module),
             "torchvision": tv, "torchvision.transforms": tv.transforms}
    sys.path.insert(0, REF_ROOT)
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update({k: v for k, v in stubs.items() if k not in sys.modules or k in ("timm", "pytorch_lightning")})
    try:
        import importlib
        return importlib.import_module("lightning.network")
    finally:
        sys.path.remove(REF_ROOT)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def cpu(out):
    import test_decoder_layout as TD
    import test_epilogue as TE
    import test_loss as TL
    save = functools.partial(save_reference, out_dir=out)

    # test_decoder_layout: Decoder.forward_coarse + Network.get_offseted_pt with an identity MLP
    net = _reference_network()
    feats, centers_grid, K, sh_dim, opacity_shift, scaling_shift = TD.decoder_inputs()
    dec = net.Decoder.__new__(net.Decoder)
    torch.nn.Module.__init__(dec)
    dec.K, dec.sh_dim, dec.opacity_dim, dec.scaling_dim, dec.rotation_dim = K, sh_dim, 1, 2, 4
    dec.mlp_coarse = torch.nn.Identity()
    r = dec.forward_coarse(feats, opacity_shift, scaling_shift)        # offset, sh, scaling, rotation, opacity
    fake_self = types.SimpleNamespace(scene_size=1.0, n_offset_groups=16, group_centers=centers_grid)
    centers = net.Network.get_offseted_pt(fake_self, r[0], K)
    save("decoder_layout", exact={"0": centers, **{str(i): t for i, t in enumerate(r[1:], 1)}})

    # test_loss: Losses.forward with a stand-in MS_SSIM that returns 1
    stub = types.ModuleType("pytorch_msssim")

    class MS_SSIM(torch.nn.Module):
        def __init__(self, **kw):
            super().__init__()

        def forward(self, a, b):
            return torch.ones((), dtype=a.dtype)
    stub.MS_SSIM = MS_SSIM
    mod = _module(os.path.join(REF_ROOT, "lightning", "loss.py"), "ref_lara_loss", {"pytorch_msssim": stub})
    for it in TL.ITERATIONS:
        out, tar = TL._fake_outputs(2, 3, 16, 24, 0)
        la = {k: v.clone().requires_grad_(k != "acc_map") for k, v in out.items()}
        loss, stats = mod.Losses()({"tar_rgb": tar}, la, it)
        loss.backward()
        exact = {"loss": loss.reshape(())}
        exact.update({"stat." + k: v.reshape(-1) for k, v in stats.items()})
        exact.update({"grad." + k: v.grad for k, v in la.items() if v.grad is not None})
        save(f"loss-{it}", exact=exact, scalars={"no_grad": ",".join(sorted(k for k, v in la.items() if v.grad is None))})

    # test_epilogue: Renderer.render_img with a stand-in rasterizer returning fixed tensors
    mod = _module(os.path.join(REF_ROOT, "lightning", "renderer_2dgs.py"), "ref_renderer_2dgs_epi")
    for depth_ratio in TE.DEPTH_RATIOS:
        color, allmap, rays, vm = TE._inputs(24, 40, 0)

        class FakeRasterizer:
            def __call__(self, **kw):
                return color, torch.zeros(kw["means3D"].shape[0], dtype=torch.int32), allmap
        r = mod.Renderer(sh_degree=1)
        r.set_rasterizer = lambda cam, device="cpu": FakeRasterizer()
        P = 5
        o = r.render_img(types.SimpleNamespace(world_view_transform=vm), rays, torch.zeros(P, 3), torch.zeros(P, 4, 3),
                         torch.zeros(P, 1), torch.zeros(P, 2), torch.randn(P, 4), "cpu", depth_ratio=depth_ratio)
        save(f"epilogue_torch-{depth_ratio}", exact=o, scalars={"keys": ",".join(sorted(o))})


if __name__ == "__main__":
    {"cpu": cpu, "gpu": gpu}[sys.argv[1]](sys.argv[2])
