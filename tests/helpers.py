"""Shared test helpers (not a test module)."""
from __future__ import annotations

import glob
import hashlib
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REFERENCE_DIR = os.path.join(GOLDEN_DIR, "reference")


def golden_files():
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def fingerprint(a) -> str:
    """Shape + SHA-256 of the bits: equal fingerprints <=> bit-identical arrays (integers compared as int64)."""
    a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a)
    if a.dtype.kind in "iub":
        a = a.astype(np.int64)
    return f"{a.dtype.str}{a.shape}:" + hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def save_reference(name, exact=None, close=None, scalars=None, k=256, out_dir=REFERENCE_DIR):
    """Stores the outputs of the unmodified reference for one test case as tests/golden/reference/<name>.npz:
    arrays a test compares bit for bit as fingerprints; arrays it compares within a tolerance relative to their
    maximum as that maximum plus a fixed, seeded sample of k non-zero elements and the largest one; scalars as is."""
    exact, close = exact or {}, close or {}
    z = {"exact.keys": np.array(list(exact), dtype=bytes), "exact.sha": np.array([fingerprint(a) for a in exact.values()], dtype=bytes),
         "close.keys": np.array(list(close), dtype=bytes)}
    idxs, vals, scales, sizes = [], [], [], []
    for a in close.values():
        a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a, dtype=np.float32).reshape(-1)
        nz = np.flatnonzero(a)
        pick = np.random.default_rng(0).choice(nz, min(k, nz.size), replace=False) if nz.size else nz
        idx = np.unique(np.append(pick, np.argmax(np.abs(a)))).astype(np.int64)
        idxs.append(idx); vals.append(a[idx])
        scales.append(np.abs(a).max() if a.size else 0.0); sizes.append(a.size)
    z["close.count"] = np.array([len(i) for i in idxs], dtype=np.int64)
    z["close.idx"] = np.concatenate(idxs) if idxs else np.zeros(0, np.int64)
    z["close.val"] = np.concatenate(vals) if vals else np.zeros(0, np.float32)
    z["close.scale"], z["close.size"] = np.array(scales, dtype=np.float64), np.array(sizes, dtype=np.int64)
    for key, v in (scalars or {}).items():
        z[key] = np.asarray(v)
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, name + ".npz"), **z)


class Reference:
    """What save_reference stored for one test case."""

    def __init__(self, name):
        with np.load(os.path.join(REFERENCE_DIR, name + ".npz")) as z:
            self.z = {k: z[k] for k in z.files}
        self.sha = dict(zip(self.z["exact.keys"].astype(str), self.z["exact.sha"].astype(str)))
        ends = np.cumsum(self.z["close.count"])
        self.close = {k: (self.z["close.idx"][e - n:e], self.z["close.val"][e - n:e], s, int(size)) for k, n, e, s, size in
                      zip(self.z["close.keys"].astype(str), self.z["close.count"], ends, self.z["close.scale"], self.z["close.size"])}

    def __getitem__(self, key):
        return self.z[key].item()

    def equal(self, key, mine) -> bool:
        return fingerprint(mine) == self.sha[key]

    def rel_err(self, key, mine) -> float:
        """rel_err(mine, reference) over the stored sample, relative to the reference's maximum."""
        idx, val, scale, size = self.close[key]
        mine = np.asarray(mine.detach().cpu() if isinstance(mine, torch.Tensor) else mine, dtype=np.float64).reshape(-1)
        assert mine.size == size, (key, mine.size)
        d = float(np.abs(mine[idx] - val).max(initial=0.0))
        return d / (scale if scale > 0 else 1.0)


def rel_err(a, b) -> float:
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if a.size == 0:
        return 0.0
    m = np.abs(b).max()
    return float(np.abs(a - b).max() / (m if m > 0 else 1.0))


def to_dev(sc, dev):
    return {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in sc.items()}


def tile_pixel_mask(ranges, H, W):
    """[H,W] bool: pixel lies in a tile whose range is non-empty (the reference leaves the median
    contributor plane uninitialised for empty tiles)."""
    gx = (W + 15) // 16
    nonempty = (ranges[:, 1] > ranges[:, 0])
    ty = np.arange(H) // 16
    tx = np.arange(W) // 16
    return nonempty[(ty[:, None] * gx + tx[None, :])]


def run_candidate(sc, cam, bg, dev, grads=None, debug=False):
    """Candidate forward (+ backward if grads=(gc,ga)) through the raw API; returns a dict of
    CPU numpy arrays including the internal state."""
    from lara_b200 import rasterizer as R
    from lara_b200 import scene as S
    from lara_b200.debug import unpack_state
    scd = to_dev(sc, dev)
    st = S.settings_for(cam, bg, sc["sh_degree"], dev, R.GaussianRasterizationSettings, debug=debug)
    H, W = cam.image_height, cam.image_width
    P = sc["means3D"].shape[0]
    color, allmap, radii, state = R.forward_raw(scd["means3D"], scd.get("shs"), scd.get("colors_precomp"),
                                                scd["opacities"], scd["scales"], scd["rotations"], None, st)
    torch.cuda.synchronize()
    u = unpack_state(state, P, H, W)
    out = {"color": color, "allmap": allmap, "radii": radii, "num_rendered": state.num_rendered}
    out.update({k: u[k] for k in ("ranges", "point_list", "n_contrib", "accum")})
    if P > 0:
        out.update({k: u[k] for k in ("tiles_touched", "depths", "transMat", "means2D", "rgb", "normal")})
    if grads is not None:
        gc, ga = grads
        g = R.backward_raw(state, radii, scd["means3D"], scd.get("shs"), scd.get("colors_precomp"), scd["scales"],
                           scd["rotations"], None, st, gc.to(dev), ga.to(dev))
        torch.cuda.synchronize()
        out.update({"g_" + k: v for k, v in g.items() if v is not None})
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in out.items()}


def scene_from_golden(z):
    sc = {"means3D": torch.from_numpy(z["means3D"]), "scales": torch.from_numpy(z["scales"]),
          "rotations": torch.from_numpy(z["rotations"]), "opacities": torch.from_numpy(z["opacities"]),
          "shs": torch.from_numpy(z["shs"]), "sh_degree": int(z["sh_degree"])}
    from lara_b200.scene import Camera
    cam = Camera(int(z["H"]), int(z["W"]), float(z["tanfovx"]), float(z["tanfovy"]),
                 torch.from_numpy(z["viewmatrix"]), torch.from_numpy(z["projmatrix"]), torch.from_numpy(z["campos"]),
                 torch.eye(4))
    return sc, cam, torch.from_numpy(z["bg"])
