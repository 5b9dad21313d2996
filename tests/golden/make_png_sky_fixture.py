"""Generates tests/golden/png_sky_rows.json from the reference's only result-bearing artefact,
rtiow_part1_final.png of Druthyn/rtiow (1200x800 RGBA8):

    python tests/golden/make_png_sky_fixture.py path/to/rtiow_part1_final.png

The scene in that render is random (main.rs:60), but pixels that only see sky are a deterministic function of
Camera::new (camera.rs:17-45) + the miss branch of ray_color (main.rs:54-56) + Color::to_rgba (vec3.rs:404-420) +
the row flip (main.rs:141-145), up to +-1 LSB of Monte-Carlo jitter inside the pixel.  We keep a grid of samples
from the top rows, which are row-uniform (no geometry reaches them).
"""
import json
import sys
from pathlib import Path

import numpy as np
from PIL import Image

SRC = Path(sys.argv[1])
OUT = Path(__file__).with_name("png_sky_rows.json")

im = np.array(Image.open(SRC))
assert im.shape == (800, 1200, 4) and (im[..., 3] == 255).all()
rows = []
for y in range(800):                      # count the leading rows with no geometry: tiny per-row spread
    if im[y, :, :3].astype(float).std(axis=0).max() > 1.5:
        break
    rows.append(y)
n_sky = len(rows)
keep_rows = list(range(0, min(n_sky, 48), 3))
keep_cols = list(range(0, 1200, 57)) + [1199]
samples = [[int(x), int(y)] + [int(c) for c in im[y, x, :3]] for y in keep_rows for x in keep_cols]
json.dump({
    "source": "rtiow_part1_final.png (Druthyn/rtiow)", "width": 1200, "height": 800,
    "camera": {"look_from": [13, 2, 3], "look_at": [0, 0, 0], "v_up": [0, 1, 0], "v_fov": 20.0, "aspect_ratio": 1.5,
               "aperture": 0.1, "focus_dist": 10.0, "cite": "main.rs:108-118"},
    "sky_only_rows": n_sky, "alpha": 255, "tolerance_lsb": 1,
    "samples_x_row_r_g_b": samples}, open(OUT, "w"))
print(f"{n_sky} sky-only rows; wrote {len(samples)} samples to {OUT}")
