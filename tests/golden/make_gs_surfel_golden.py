"""Generates tests/golden/gs_surfel_loop.npz by running the reference's UNMODIFIED
/root/reference/nsr/gs_surfel.py `GaussianRenderer2DGS.render` -- its own B x V Python loop and
post-processing (lines 41-202) -- on CPU.

The file is executed as it lies in /root/reference (importlib from its path; `nsr/__init__.py` is not run).  What
it imports but this image lacks is stubbed:
  * `diff_surfel_rasterization` (third party, not vendored): an oracle-backed module with upstream's binding
    surface -- `GaussianRasterizationSettings` NamedTuple + `GaussianRasterizer(raster_settings)(means3D=...,
    means2D=..., shs=None, colors_precomp=..., opacities=..., scales=..., rotations=..., cov3D_precomp=None)`
    -> (color[3,H,W], radii[P], allmap[7,H,W]) -- computed by oracle/surfel_oracle.c.  So the golden pins the
    reference's LOOP and POST-PROCESSING around the rasteriser; the rasteriser arithmetic itself stays
    "parity unpinned" (see oracle/surfel_oracle.c).
  * `kiui`, `point_cloud_utils`, `cv2`, `matplotlib` (never used on this path): dummies from _ref_stubs.
  * the hard-coded `device="cuda"` of its constructor (gs_surfel.py:25): torch.tensor is wrapped to place such
    tensors on the CPU while the module is constructed.
Only runs inside the build container (needs /root/reference); the .npz it writes is committed and is what
tests/test_raster_gpu.py::test_reference_loop_golden compares the CUDA mirror with.

It also writes gs_surfel_loop_calls.json: every call the reference's loop made to the rasteriser, in order -- which
batch item and view it passed (checked here to be exactly the golden's `g` / `view` / `proj` at those indices), the
background, scale modifier and image size, and sha256 digests of the raw (color, radii, allmap) the shim returned.
The golden is the reference's post-processing of exactly those returns, so tests/test_round2_cpu.py pins the golden
without the reference tree by replaying every call through the C oracle and comparing the digests.
    python tests/golden/make_gs_surfel_golden.py [--check]
"""
import hashlib
import importlib.util
import json
import os
import sys
import types
from typing import NamedTuple

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import surfel_oracle as so  # noqa: E402
from tools import synth  # noqa: E402

OUT = os.path.join(HERE, "gs_surfel_loop.npz")
CALLS = os.path.join(HERE, "gs_surfel_loop_calls.json")
_calls = []                                            # what the reference's loop passed to / got from the shim


# ---- oracle-backed stand-in for the un-vendored third-party module --------------------------------------------
class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


class GaussianRasterizer(torch.nn.Module):
    def __init__(self, raster_settings):
        super().__init__()
        self.raster_settings = raster_settings

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        assert shs is None and cov3D_precomp is None and colors_precomp is not None
        rs = self.raster_settings
        o = so.rasterize(means3D.numpy(), opacities.numpy(), scales.numpy(), rotations.numpy(), colors_precomp.numpy(),
                         rs.viewmatrix.numpy(), rs.projmatrix.numpy(), rs.bg.numpy(), int(rs.image_height),
                         int(rs.image_width), float(rs.scale_modifier))
        assert rs.image_height == rs.image_width
        _calls.append(dict(g13=torch.cat([means3D, opacities, scales, rotations, colors_precomp], 1).numpy(),
                           view=rs.viewmatrix.numpy().copy(), proj=rs.projmatrix.numpy().copy(), bg=rs.bg.numpy().copy(),
                           scale_modifier=float(rs.scale_modifier), size=int(rs.image_height),
                           color=o["color"], radii=o["radii"], allmap=o["allmap"]))
        return torch.from_numpy(o["color"]), torch.from_numpy(o["radii"]), torch.from_numpy(o["allmap"])


def load_reference_renderer():
    sys.path.insert(0, HERE)
    import _ref_stubs  # noqa: F401  (puts the reference tree on sys.path, installs the dummies)
    shim = types.ModuleType("diff_surfel_rasterization")
    shim.GaussianRasterizationSettings = GaussianRasterizationSettings
    shim.GaussianRasterizer = GaussianRasterizer
    sys.modules["diff_surfel_rasterization"] = shim
    spec = importlib.util.spec_from_file_location("ref_nsr_gs_surfel", "/root/reference/nsr/gs_surfel.py")
    mod_ = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod_)                      # the unmodified reference file
    real_tensor = torch.tensor

    def cpu_tensor(*a, **k):
        if str(k.get("device", "")).startswith("cuda"):
            k["device"] = "cpu"
        return real_tensor(*a, **k)
    torch.tensor = cpu_tensor
    try:
        rnd = mod_.GaussianRenderer2DGS(64, 3, {"z_near": 0.01})
    finally:
        torch.tensor = real_tensor
    return rnd


def cases():
    """Two calls: defaults (white bg, scale 1, ctor output size) and (bg, scale_modifier, output_size) overrides."""
    vs, ps, cs, tf = [], [], [], None
    for k in range(6):
        v, p, c, tf = synth.camera_from_pose25(synth.orbit_pose25(25.0 + 53.0 * k, 10.0 + 9.0 * (k % 3)))
        vs.append(v); ps.append(p); cs.append(c)
    cam = dict(view=np.stack(vs).reshape(2, 3, 4, 4), proj=np.stack(ps).reshape(2, 3, 4, 4),
               pos=np.stack(cs).reshape(2, 3, 3), tanfov=tf)
    g = np.stack([synth.synthetic_surfels(1200, 71, scale_boost=12.0), synth.synthetic_surfels(1200, 72, scale_boost=4.0)])
    return g, cam


def generate():
    rnd = load_reference_renderer()
    g, cam = cases()
    T = torch.from_numpy
    out = {"g": g, "view": cam["view"], "proj": cam["proj"], "pos": cam["pos"], "tanfov": np.float32(cam["tanfov"])}
    a = rnd.render(T(g), T(cam["view"]), T(cam["proj"]), T(cam["pos"]), cam["tanfov"])
    bg = torch.tensor([0.2, 0.5, 0.9])
    b = rnd.render(T(g[:1]), T(cam["view"][:1, :2]), T(cam["proj"][:1, :2]), T(cam["pos"][:1, :2]), cam["tanfov"],
                   bg_color=bg, scale_modifier=1.6, output_size=48)
    for tag, r in (("a", a), ("b", b)):
        for k, v in r.items():
            out["%s__%s" % (tag, k)] = v.numpy().astype(np.float32)
    out["b__bg"] = bg.numpy()
    return out, recorded_calls(g, cam["view"], cam["proj"])


def digest(a):
    """sha256 of an array's dtype, shape and bytes: a bit-exact pin that stays small."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()


def recorded_calls(g, view, proj):
    """The shim's record; each call is tied to the one (batch item, view) of the golden inputs it was given."""
    rec = []
    for i, c in enumerate(_calls):
        hits = [(b, v) for b in range(view.shape[0]) for v in range(view.shape[1])
                if np.array_equal(c["g13"], g[b]) and np.array_equal(c["view"], view[b, v])
                and np.array_equal(c["proj"], proj[b, v])]
        assert len(hits) == 1, (i, hits)
        rec.append({"item": hits[0][0], "view": hits[0][1], "bg": [float(x) for x in c["bg"]],
                    "scale_modifier": c["scale_modifier"], "size": c["size"],
                    "sha256": {k: digest(c[k]) for k in ("color", "radii", "allmap")}})
    return rec


if __name__ == "__main__":
    new, calls = generate()
    if "--check" in sys.argv:
        old = np.load(OUT)
        for k in new:
            assert np.array_equal(np.asarray(new[k]), old[k]), k
        with open(CALLS) as f:
            assert json.load(f) == calls, CALLS
        print("golden reproduces bit for bit:", OUT, CALLS)
    else:
        np.savez_compressed(OUT, **new)
        with open(CALLS, "w") as f:
            json.dump(calls, f, indent=1)
            f.write("\n")
        print("wrote", OUT, os.path.getsize(OUT), "bytes and", CALLS)
