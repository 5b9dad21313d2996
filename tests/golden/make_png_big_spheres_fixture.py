"""Generates tests/golden/png_big_spheres.json from the reference's only result-bearing artefact,
rtiow_part1_final.png of Druthyn/rtiow (1200x800 RGBA8):

    python tests/golden/make_png_big_spheres_fixture.py path/to/rtiow_part1_final.png

random_scene (main.rs:59-102) is random in its small spheres only: the ground (main.rs:62-64) and the three unit spheres —
glass at (0,1,0), Lambertian (0.4,0.2,0.1) at (-4,1,0), Metal (0.7,0.6,0.5) fuzz 0 at (4,1,0) (main.rs:93-99) — are fixed, and so
is the camera (main.rs:108-118).  Three regions of the reference's render therefore do not depend on the random part:

  metal  the upper cap of the metal sphere mirrors nothing but sky: Camera::get_ray -> Sphere::hit (point, normal) ->
         Metal::scatter (reflect, albedo) -> recursion -> sky -> to_rgba, exactly (only pixel jitter and the lens move a sample)
  glass  the lower part of the glass sphere shows the sky through two refractions: Dialectric::scatter (refract, Schlick);
         a few per cent of its light are reflections of the random neighbourhood
  brown  the sky-facing top of the diffuse sphere: Lambertian::scatter + albedo; the random neighbourhood only darkens it slightly

  horizon  the defocused transition from sky to the far ground, left and right of the sphere field: the f64 ground sphere
         (main.rs:62-64) hit at grazing incidence, the thin lens (camera.rs:47-54: the horizon is far out of focus) and the Lambertian
         ground under the open sky; columns are kept where the PNG shows the bare far-ground colour below the band

We keep 9x9-pixel block means (the render is converged: block std <= ~1 LSB) on a grid inside each region, selected by colour
and smoothness in the PNG itself.
"""
import json
import sys
from pathlib import Path

import numpy as np
from PIL import Image

SRC = Path(sys.argv[1])
OUT = Path(__file__).with_name("png_big_spheres.json")

im = np.array(Image.open(SRC)).astype(float)
assert im.shape == (800, 1200, 4)
REGIONS = {   # name: (x range, y range, colour predicate on the block mean, tolerance of the block mean in LSB: [lo, hi] of ours - png)
    "metal": ((590, 1040), (60, 292), lambda m: abs(m[2] - 181.0) < 0.6 and m[0] > 140, [-0.25, 0.25]),
    "glass": ((440, 610), (236, 345), lambda m: m[2] > 246 and m[0] > 195, [-1.0, 2.5]),
    "brown": ((350, 475), (66, 205), lambda m: 100 < m[0] < 130 and 80 < m[1] < 105 and 60 < m[2] < 90, [-0.5, 4.5]),
}
out = {}
for name, ((x0, x1), (y0, y1), pred, tol) in REGIONS.items():
    pts = []
    for y in range(y0, y1, 14):
        for x in range(x0, x1, 14):
            blk = im[y - 4:y + 5, x - 4:x + 5, :3].reshape(-1, 3)
            m, s = blk.mean(0), blk.std(0)
            if s.max() < 1.3 and pred(m):
                pts.append([x, y] + [round(float(c), 3) for c in m])
    out[name] = {"tolerance_lsb_lo_hi": tol, "half_w": 4, "half_h": 4, "blocks_x_y_r_g_b": pts}
    if name == "metal":
        out[name]["max_abs_mean"] = 0.1          # no bias at all: mean over the blocks of (ours - png), per channel
    print(name, len(pts), "blocks")
# horizon band: 15x3 blocks (the band is row-uniform locally) in columns whose row 200 shows the bare far ground
pts = []
FAR_GROUND = np.array([137.8, 156.1, 181.0])
for x in list(range(15, 330, 35)) + list(range(1080, 1190, 35)):
    if np.abs(im[199:202, x - 7:x + 8, :3].reshape(-1, 3).mean(0) - FAR_GROUND).max() > 0.4:
        continue
    for y in range(166, 202, 3):
        blk = im[y - 1:y + 2, x - 7:x + 8, :3].reshape(-1, 3)
        if blk.std(0).max() < 6.0:           # the band itself has a vertical gradient of ~5 LSB per row
            pts.append([x, y] + [round(float(c), 3) for c in blk.mean(0)])
out["horizon"] = {"tolerance_lsb_lo_hi": [-2.5, 2.5], "max_abs_mean": 0.4, "half_w": 7, "half_h": 1, "blocks_x_y_r_g_b": pts}
print("horizon", len(pts), "blocks")
json.dump({
    "source": "rtiow_part1_final.png (Druthyn/rtiow)", "width": 1200, "height": 800, "block": 9,
    "camera": {"look_from": [13, 2, 3], "look_at": [0, 0, 0], "v_up": [0, 1, 0], "v_fov": 20.0, "aspect_ratio": 1.5,
               "aperture": 0.1, "focus_dist": 10.0, "cite": "main.rs:108-118"},
    "scene": {"cite": "main.rs:62-64,93-99 (the non-random part of random_scene)",
              "center": [[0, -1000, 0], [0, 1, 0], [-4, 1, 0], [4, 1, 0]], "radius": [1000, 1, 1, 1],
              "mat_kind": [0, 2, 0, 1], "mat_albedo": [[0.5, 0.5, 0.5], [1, 1, 1], [0.4, 0.2, 0.1], [0.7, 0.6, 0.5]], "mat_param": [0, 1.5, 0, 0]},
    "regions": out}, open(OUT, "w"))
print("wrote", OUT)
