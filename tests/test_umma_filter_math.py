"""CPU restatement of the tensor-core sphere filter's arithmetic (rtiow_b200/csrc/rt_umma.cuh, capi.cu's feature image).

The filter decides `discriminant >= 0` of sphere.rs:18-25 for every (ray, sphere) pair as one contraction
D = row1 . B1^T + row2 . B2^T of fp16 operands (hi/lo split of 11 features per side, K slots shared between the three products).
This file restates, in numpy, exactly what the CUDA side does — feature values, power-of-two scales, the fp16 split, the slot
map of `umma::ray_rows` / `umma::b2_feature`, the order of the two products with an fp16 rounding of the intermediate and of the
result — and checks on the final scene (main.rs:59-102) that
  * the contraction reproduces the f64 discriminant to within a fraction of the slack folded into S_0,
  * no sphere with discriminant >= 0 is ever filtered out (the filter is a conservative superset),
  * padding entries and "dead" rows (a line that misses the scene's bounding sphere) can never pass,
  * the column permutation `umma::d16_column` is the inverse of the bit order the packed sign collection returns.
No GPU and no library call besides the seeded scene generator: the GPU counterpart is tests/test_tensor_scan_gpu.py
(bit-identical hits from the FP32 and the tensor filter) and tools/probe_umma_filter.cu (the same error measured on the B200).
"""
import numpy as np
import pytest

import scan_scenes
from test_parity_unit_gpu import f32_scene

f16, f32 = np.float16, np.float32


def split(x):
    """x (f32) = hi + lo, two fp16 (cvt.rn.f16.f32 of x and of the remainder)"""
    x = np.asarray(x, f32)
    hi = x.astype(f16)
    lo = (x - hi.astype(f32)).astype(f16)
    return hi, lo


def b2_feature(blk, s):
    """umma::b2_feature: K slot s of B block blk holds feature `feat` of the sphere, its lo part when is_lo"""
    if blk == 0:
        return (s if s < 10 else 10 if s < 12 else s - 12), False
    return (s if s < 10 else s - 6), s < 10


def ray_rows(f, d, live, sigma, sc):
    """umma::ray_feature_values + umma::ray_rows, in f32 like the device code; f, d: [n, 3]"""
    f = f.astype(f32); d = d.astype(f32)
    s0, s1, s4, s10 = (f32(v) for v in sc)
    a = (d * d).sum(1, dtype=f32)
    fd = (f * d).sum(1, dtype=f32)
    R = np.zeros((len(f), 12), f32)
    R[:, 0] = a * s0
    R[:, 1:4] = (a[:, None] * f - fd[:, None] * d) * (f32(2) * s1)
    R[:, 4:7] = d * d * s4
    R[:, 7] = d[:, 0] * d[:, 1] * (f32(2) * s4); R[:, 8] = d[:, 0] * d[:, 2] * (f32(2) * s4); R[:, 9] = d[:, 1] * d[:, 2] * (f32(2) * s4)
    R[:, 10] = (fd * fd - a * (f * f).sum(1, dtype=f32) + f32(sigma)) * s10
    R[~live, :10] = 0; R[~live, 10] = -1
    hi, lo = split(R)
    row1 = np.concatenate([hi[:, :10], hi[:, 10:11], lo[:, 10:11], lo[:, 0:4]], 1)      # [ hi_0..9 | hi_10 lo_10 | lo_0..3 ]
    row2 = np.concatenate([hi[:, :10], lo[:, 4:10]], 1)                                 # [ hi_0..9 | lo_4..9 ]
    assert row1.shape[1] == row2.shape[1] == 16
    return row1, row2


def sphere_image(center, radius, npad, R_scene, sc, bypass=False):
    """capi.cu: the 11 sphere features (f64 -> f32 -> fp16 hi/lo) in the two K = 16 blocks, padding entries never pass.
    bypass (rtiow_ctx_set_filter_bypass): every real column is S_0 = Rp^2 / s0, S_10 = -1 / s10 and zeros, and passes every ray"""
    s0, s1, s4, s10 = sc
    Rp = 2.0 ** np.ceil(np.log2(R_scene))
    slack = 1.5625e-5 * R_scene * R_scene
    c = center.astype(f32).astype(np.float64); r = radius.astype(f32).astype(np.float64)      # the f32 sphere the precise test sees
    S = np.zeros((npad, 11))
    n = len(c)
    S[:n, 0] = (r * r - (c * c).sum(1) + slack) / s0
    S[:n, 1:4] = c / s1
    S[:n, 4:7] = c * c / s4
    S[:n, 7] = c[:, 0] * c[:, 1] / s4; S[:n, 8] = c[:, 0] * c[:, 2] / s4; S[:n, 9] = c[:, 1] * c[:, 2] / s4
    S[n:, 0] = -2.0 * Rp * Rp / s0      # padding: D = -2 Rp^2 - |f|^2 (+ sigma), |D| <= 2 Rp^2 + R^2 < 65504 wherever d_fits holds
    S[:, 10] = 1.0 / s10
    if bypass:
        S[:n] = 0.0
        S[:n, 0] = Rp * Rp / s0; S[:n, 10] = -1.0 / s10
    hi, lo = split(S.astype(f32))
    assert not lo[:, 10].any(), "S_10 is a power of two: the two-product form relies on its lo part being zero"
    B = np.zeros((2, npad, 16), f16)
    for blk in range(2):
        for s in range(16):
            feat, is_lo = b2_feature(blk, s)
            B[blk, :, s] = (lo if is_lo else hi)[:, feat]
    return B, slack


def contraction(row1, row2, B):
    """two tcgen05.mma kind::f16 with an fp16 accumulator: products exact, sums in f32, the intermediate D and the result rounded to fp16"""
    d_cross = (row2.astype(f32) @ B[1].astype(f32).T).astype(f16)                      # row2 . B2: cross terms only
    return (row1.astype(f32) @ B[0].astype(f32).T + d_cross.astype(f32)).astype(f16)    # + row1 . B1: all of hi.hi, rounded once


def test_two_product_form_covers_every_term_once():
    """hi.hi (11) + hi.lo (10: S_10 has no lo part) + lo.hi (11) = 32 terms = the 2 x 16 K slots, each exactly once"""
    terms = []
    ray = {0: [("hi", k) for k in range(10)] + [("hi", 10), ("lo", 10)] + [("lo", k) for k in range(4)],
           1: [("hi", k) for k in range(10)] + [("lo", k) for k in range(4, 10)]}
    for blk in range(2):
        for s in range(16):
            feat, is_lo = b2_feature(blk, s)
            part, k = ray[blk][s]
            assert k == feat, "ray slot and sphere slot carry the same feature"
            terms.append((part, "lo" if is_lo else "hi", feat))
    want = [("hi", "hi", k) for k in range(11)] + [("hi", "lo", k) for k in range(10)] + [("lo", "hi", k) for k in range(11)]
    assert sorted(terms) == sorted(want) and len(set(terms)) == 32


def test_d16_column_inverts_the_packed_sign_order():
    """umma::sign_word16 returns bit 8 b + j = sign of column 4 j + b; umma::d16_column(k) must put sphere k where bit 31 - k reads"""
    d16_column = lambda k: 4 * ((31 - k) & 7) + ((31 - k) >> 3)
    cols = [d16_column(k) for k in range(32)]
    assert sorted(cols) == list(range(32))
    for k, col in enumerate(cols):
        j, b = col // 4, col % 4
        assert 8 * b + j == 31 - k


def restate(c, r, o, d, bypass=False):
    """the filter of closest_hit_umma on the small spheres (c, r) and unit rays (o, d), all f32 values:
    -> D [rays, npad] (the contraction, f64 copy), the f64 discriminant [rays, ns], live rows, slack, R.
    With bypass the image is rtiow_ctx_set_filter_bypass's and the rows carry the device's per-ray sigma."""
    R_scene = max(1.0, float((np.linalg.norm(c, axis=1) + np.abs(r)).max()))
    Rp = 2.0 ** np.ceil(np.log2(R_scene))
    sc = (Rp, 1.0, Rp * 0.5, 1.0 / Rp)                                        # umma::FeatScale {s0, s1, s4, s10}
    npad = -(-len(c) // 64) * 64
    B, slack = sphere_image(c, r, npad, R_scene, sc, bypass)
    # line_gate (rt_scene.cuh): foot point of the coordinate origin (orthogonalised twice), liveness against the bounding sphere
    a = (d * d).sum(1)
    f = o - d * ((o * d).sum(1) / a)[:, None]
    f = f - d * ((f * d).sum(1) / a)[:, None]
    sigma = scan_scenes.SIGMA_PER_LEN * max(float(np.abs(r).max()), 1e-3) * np.abs(o).sum(1) if bypass else 0.0
    live = (f * f).sum(1) < R_scene * R_scene * (1 + 1e-6) + sigma
    row1, row2 = ray_rows(f, d, live, sigma, sc)
    D = contraction(row1, row2, B).astype(np.float64)
    oc = c[None, :, :].astype(f32).astype(np.float64) - o[:, None, :]
    hb = (oc * d[:, None, :]).sum(2)
    disc = hb * hb - a[:, None] * ((oc * oc).sum(2) - (r.astype(f32).astype(np.float64) ** 2)[None, :])        # sphere.rs:24 (quarter form)
    return D, disc, live, slack, R_scene


def test_contraction_reproduces_the_discriminant_and_never_drops_a_hit(capi):
    scene = capi.random_scene(1)
    small = np.abs(scene["radius"]) <= 8.0                                     # the r = 1000 ground goes to the large-sphere test
    c, r = scene["center"][small], scene["radius"][small]

    rng = np.random.default_rng(7)
    n = 4096
    # camera rays from (13, 2, 3) and bounce rays leaving points of the sphere field, plus rays that miss the scene entirely
    o = np.where(rng.random((n, 1)) < 0.4, np.array([13.0, 2.0, 3.0]) + 0.05 * rng.standard_normal((n, 3)),
                 np.stack([24 * (rng.random(n) - 0.5), 0.4 * rng.random(n), 24 * (rng.random(n) - 0.5)], 1))
    t = np.stack([22 * (rng.random(n) - 0.5), 3 * rng.random(n) - 0.5, 22 * (rng.random(n) - 0.5)], 1)
    d = t - o
    d[-256:] = np.array([0.0, 1.0, 0.0]) + 0.01 * rng.standard_normal((256, 3)); o[-256:, 0] += 60.0       # far outside, heading up
    o = o.astype(f32).astype(np.float64)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32).astype(np.float64)
    a = (d * d).sum(1)

    D, disc, live, slack, R_scene = restate(c, r, o, d)
    assert live[:-256].mean() > 0.9 and not live[-256:].any()
    nreal = len(c)
    # 1. padding and dead rows never pass
    assert (D[:, nreal:] < 0).all()
    assert (D[~live] < 0).all()
    # 2. where the sign is decided, the contraction is the discriminant + slack to a fraction of the slack
    want = disc[live] + slack * a[live, None]
    near = np.abs(want) < 0.05
    err = np.abs(D[live][:, :nreal] - want)[near]
    assert err.max() < 0.25 * slack, (err.max(), slack)
    # 3. conservative: every sphere the exact test could accept passes; few others do
    hit = disc[live] >= 0
    passed = D[live][:, :nreal] >= 0
    assert not (hit & ~passed).any(), "the filter dropped a sphere whose discriminant is >= 0"
    assert passed.sum() <= 1.25 * hit.sum()
    # 4. a ray that hits nothing far away still cannot overflow the fp16 result: |D| <= 4 R^2 << 65504
    assert np.isfinite(D).all() and 4 * R_scene * R_scene < 60000


def _unit_f32(d):
    return (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32).astype(np.float64)


def _chunks(o, d, n=2048):
    for s in range(0, len(o), n):
        yield o[s:s + n], d[s:s + n]


def _boundary_scene(capi, name):
    arrays = scan_scenes.sparse_ball(122.4) if name == "ball-R122.4" else scan_scenes.build(name, capi)
    info = scan_scenes.scene_info(arrays)
    assert info["failing"] == [], info["failing"]
    return arrays, info


def test_contraction_drops_no_hit_at_silhouettes(capi):
    """the final scene's rays grazing sphere silhouettes (scan_scenes.silhouette_rays), inside the band where the split and the
    fp16 accumulation decide: nothing with discriminant >= 0 is dropped, and the contraction tracks disc + slack there too"""
    scene = f32_scene(capi.random_scene(1))
    small = np.abs(scene["radius"]) <= 8.0
    c, r = scene["center"][small], scene["radius"][small]
    o, d, target = scan_scenes.silhouette_rays(scene)
    scan_scenes.assert_band_coverage(scene, o, d, target)
    d = _unit_f32(d)
    for oo, dd in _chunks(o, d):
        D, disc, live, slack, _ = restate(c, r, oo, dd)
        hit = disc >= 0
        assert not (hit & live[:, None] & (D[:, :len(c)] < 0)).any(), "the filter dropped a sphere whose discriminant is >= 0"
        assert not (hit & ~live[:, None]).any(), "a line the gate calls dead meets a sphere"
        want = disc[live] + slack * (dd * dd).sum(1)[live, None]
        near = np.abs(want) < 0.05
        assert np.abs(D[live][:, :len(c)] - want)[near].max() < 0.25 * slack
        assert np.isfinite(D).all()


@pytest.mark.parametrize("name", ["ball-R122.4", "compact-3137", "row-r0.4"])
def test_contraction_at_the_selection_boundaries(capi, name):
    """the scenes at the edges of the tensor filter's rules (tests/scan_scenes.py): R just under 122.47 (Rp = 128, 4 R^2 just
    under 60000, padding columns past the last word of small spheres), the largest image (npad 3200, 63 padding columns), and
    the slack just below the mean r^2, on scan_scenes.rays and the silhouette rays.  No sphere with discriminant >= 0 is
    dropped, every column of every ray stays finite in fp16, and the padding columns stay negative."""
    arrays, info = _boundary_scene(capi, name)
    k = info["small"]
    c, r = arrays["center"][k], arrays["radius"][k]
    o, d = scan_scenes.rays(name, arrays)
    o2, d2, _ = scan_scenes.silhouette_rays(arrays)
    o, d = np.concatenate([o, o2]), _unit_f32(np.concatenate([d, d2]))
    ns = len(c)
    n_live = 0
    for oo, dd in _chunks(o, d):
        D, disc, live, _, _ = restate(c, r, oo, dd)
        n_live += live.sum()
        assert not ((disc >= 0) & live[:, None] & (D[:, :ns] < 0)).any(), "the filter dropped a sphere whose discriminant is >= 0"
        assert np.isfinite(D[:, :ns]).all()
        pad = D[:, ns:]
        assert pad.shape[1] == info["npad"] - ns > 0
        assert np.isfinite(pad).all(), f"{(~np.isfinite(pad)).sum()} padding entries overflow fp16"
        assert (pad < 0).all()
    assert n_live > 0.5 * len(o)


@pytest.mark.parametrize("name", ["ball-R122.4", "compact-3137"])
def test_bypass_image_passes_every_sphere(capi, name):
    """rtiow_ctx_set_filter_bypass's tensor image: every real column passes (sign bit clear) on live and dead rows alike, no
    padding column ever passes, and every entry is finite in fp16 — at Rp = 128 (the largest |D|) and with 63 padding columns"""
    arrays, info = _boundary_scene(capi, name)
    k = info["small"]
    c, r = arrays["center"][k], arrays["radius"][k]
    o, d = scan_scenes.rays(name, arrays)
    o2, d2, _ = scan_scenes.silhouette_rays(arrays)
    o, d = np.concatenate([o, o2]), _unit_f32(np.concatenate([d, d2]))
    ns = len(c)
    n_live = n_dead = 0
    for oo, dd in _chunks(o, d):
        D, _, live, _, _ = restate(c, r, oo, dd, bypass=True)
        n_live += live.sum(); n_dead += (~live).sum()
        assert np.isfinite(D).all()
        assert not np.signbit(D[:, :ns]).any(), f"{np.signbit(D[:, :ns]).sum()} real columns do not pass"
        assert np.signbit(D[:, ns:]).all() and info["npad"] > ns
    assert n_live > 1000 and n_dead > 100, (n_live, n_dead)
