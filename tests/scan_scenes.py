"""Scenes, rays and a host-logic mirror for testing every arm of the F32 hit scan (test infrastructure, not a test file).

`plan_scan` (rtiow_b200/csrc/capi.cu) sends each scan to one of five arms: Tensor (the tcgen05 filter), Smem, Wide and Global
(the FP32 filter with its table in 48 KB of shared memory, in one wide CTA, or read from global memory) and F64.  Which one
depends on the scene, so a test that runs on whatever SCAN_AUTO picks may not exercise the code it was written for.
`scan_arm` restates the host rules in numpy:
  * the small / big split of rtiow_scene_upload (|r| > 8 or reach > 4096 -> the f64 list of large spheres),
  * the rules of tensor_image (the tensor filter's image must fit shared memory, its slack must stay below the mean r^2, and
    the fp16 accumulator must stay finite),
  * plan_scan (FP32 table size against the shared memory of a 256-thread CTA and of one wide 512-thread CTA).
`SCENES` lists seeded scenes whose sizes sit on both sides of each rule, with the arm each backend must select.
`robust_closest` is the f64 closest hit over every sphere, with the second-closest root, so that a test can demand an exact
index wherever the answer is not a knife edge.
"""
import math
import re
from functools import lru_cache
from pathlib import Path

import numpy as np

from rtiow_b200.capi import F32, F64, SCAN_AUTO, SCAN_FP32, SCAN_TENSOR
from test_parity_unit_gpu import f32_scene, not_grazing

CSRC = Path(__file__).resolve().parent.parent / "rtiow_b200" / "csrc"


def _define(header, name):
    m = re.search(rf"^\s*#define\s+{name}\s+(\d+)\b", (CSRC / header).read_text(), re.M)
    assert m, f"{name} not found in {header}"
    return int(m.group(1))


CAND_CAP = _define("rt_scene.cuh", "RT_CAND_CAP")              # uint16 candidate slots per lane
UMMA_GROUPS = _define("rt_umma_scan.cuh", "RT_UMMA_GROUPS")    # ray groups of 128 per tensor CTA
UMMA_CHUNK = _define("rt_umma_scan.cuh", "RT_UMMA_CHUNK")      # spheres per MMA chunk: the image pads to a multiple of it
SMEM_CTA = 227 * 1024          # plan_scan / tensor_image: the most shared memory one CTA may have on sm_100
SMEM_SMALL = 56 * 1024         # plan_scan: the FP32 table + 256 lists fit three 256-thread CTAs per SM (Smem)
BIG_RADIUS, BIG_REACH = 8.0, 4096.0                            # rtiow_scene_upload: kBigRadius, and the reach of a small sphere

ARMS = ("Tensor", "Smem", "Wide", "Global", "F64")


def umma_smem_bytes(npad):
    """UmmaShape<G, NC>::smem_bytes: candidate lists, the two fp16 K blocks of npad spheres (32 bytes each), mbarriers"""
    cand = UMMA_GROUPS * 128 * CAND_CAP * 2
    need = ((cand + 127) & ~127) + 2 * npad * 32 + UMMA_GROUPS * 8 * 8 + 16 + UMMA_GROUPS * 4
    return max(need, 120 * 1024)


def scene_info(arrays):
    """what rtiow_scene_upload derives from a scene: the small spheres, their padded counts, R and the tensor rules that fail"""
    c = np.asarray(arrays["center"], float).reshape(-1, 3); r = np.asarray(arrays["radius"], float)
    reach = np.sqrt((c * c).sum(1)) + np.abs(r)
    small = ~((np.abs(r) > BIG_RADIUS) | (reach > BIG_REACH))
    cs = c[small].astype(np.float32).astype(float); rs = r[small].astype(np.float32).astype(float)       # the f32 copy in `small`
    ns = int(small.sum())
    np_ = -(-ns // 32) * 32
    npad = -(-ns // UMMA_CHUNK) * UMMA_CHUNK
    R = max(1.0, float((np.sqrt((cs * cs).sum(1)) + np.abs(rs)).max())) if ns else 1.0
    Rp = 2.0 ** math.ceil(math.log2(R))
    slack = 1.5625e-5 * R * R
    mean_r2 = float((rs * rs).mean()) if ns else 0.0
    rules = {
        "empty": ns > 0,
        "npad": npad < 65536,
        "smem": umma_smem_bytes(npad) <= SMEM_CTA,
        "reach": Rp <= 8192.0,
        "slack": slack <= mean_r2,
        "d_fits": 4.0 * R * R < 60000.0,
    }
    return dict(small=np.flatnonzero(small), ns=ns, np=np_, npad=npad, R=R, Rp=Rp, slack=slack, mean_r2=mean_r2,
                failing=[k for k, ok in rules.items() if not ok])


def scan_arm(arrays, backend=SCAN_AUTO, precision=F32):
    """-> (arm, failing tensor rules).  arm is None where plan_scan refuses (TENSOR forced on a scene that does not qualify)."""
    info = scene_info(arrays)
    failing = info["failing"]
    if precision == F64:
        return "F64", failing
    if not failing and backend != SCAN_FP32:
        return "Tensor", failing
    if backend == SCAN_TENSOR:
        return None, failing
    table = (4 * info["np"] + 16) * 4                    # RT_TABLE_FLOATS(np) floats
    if table + 256 * CAND_CAP * 2 <= SMEM_SMALL:
        return "Smem", failing
    if table + 512 * CAND_CAP * 2 <= SMEM_CTA:
        return "Wide", failing
    return "Global", failing


# ------------------------------------------------------------------------------------------------ scene builders
def _materials(n, rng):
    """one material per sphere: Lambertian, Metal or Dielectric, as random_scene mixes them"""
    kind = rng.choice([0, 1, 2], n, p=[0.6, 0.25, 0.15]).astype(np.uint32)
    param = np.where(kind == 1, rng.uniform(0, 0.5, n), 1.5)
    return dict(mat_index=np.arange(n, dtype=np.uint32), mat_kind=kind, mat_albedo=rng.uniform(0.1, 0.95, (n, 3)),
                mat_param=param)


def _scene(center, radius, rng, exact=False):
    """shuffled into a random list order (a filter that scans positions in order then cannot hide a lost candidate behind
    the geometry), f32-rounded unless `exact`"""
    perm = rng.permutation(len(radius))
    arrays = dict(center=np.asarray(center, float).reshape(-1, 3)[perm], radius=np.asarray(radius, float)[perm],
                  **_materials(len(radius), rng))
    return arrays if exact else f32_scene(arrays)


def _lattice_points(n, spacing, rng, jitter=0.05, exclude=None):
    """the n points of a cubic lattice nearest the coordinate origin, each moved by up to jitter * spacing per axis"""
    k = int(math.ceil((n * 6 / math.pi) ** (1 / 3) / 2)) + 3
    g = np.arange(-k, k + 1, dtype=float)
    p = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) * spacing
    if exclude is not None:
        p = p[~exclude(p)]
    p = p[np.argsort(np.linalg.norm(p, axis=1), kind="stable")[:n]]
    assert len(p) == n
    return p + rng.uniform(-jitter, jitter, p.shape) * spacing


def compact(ns, seed=0):
    """ns non-overlapping spheres (r 0.1 .. 0.6) on a jittered lattice of spacing 1.5: R ~ 10 at 1 000 spheres"""
    rng = np.random.default_rng(1000 + ns + seed)
    return _scene(_lattice_points(ns, 1.5, rng), rng.uniform(0.1, 0.6, ns), rng)


def row(r, n=200, spacing=0.5, seed=0):
    """n spheres of radius r on the x axis from 0 to (n - 1) spacing: R ~ 100 (the slack rule's boundary sits at r ~ 0.39)"""
    rng = np.random.default_rng(2000 + seed)
    c = np.stack([np.arange(n) * spacing, np.zeros(n), np.zeros(n)], 1)
    return _scene(c, np.full(n, r), rng)


def sparse_ball(R, ns=985, seed=0):
    """a cluster of ns - 1 spheres with radii 0.7 .. 0.9 on a lattice of spacing 2 around the coordinate origin, and one sphere
    whose far side is R from it: R sets Rp and the fp16 range of the tensor filter without changing anything else"""
    rng = np.random.default_rng(3000 + seed)
    c = _lattice_points(ns - 1, 2.0, rng)
    u = np.array([1.0, 0.3, -0.5]) / np.linalg.norm([1.0, 0.3, -0.5])
    c = np.concatenate([c, [u * (R - 0.8)]]); r = np.concatenate([rng.uniform(0.7, 0.9, ns - 1), [0.8]])
    return _scene(c, r, rng)


def field_row(seed=0):
    """41 overlapping spheres of radius 0.3 every 0.5 along the x axis from -10 to 10, in a field of 400 spheres that keeps
    the scene on the tensor filter (R ~ 10.3): a ray along the row has ~40 spheres with disc >= 0, past RT_CAND_CAP"""
    rng = np.random.default_rng(4000 + seed)
    x = np.arange(-20, 21) * 0.5
    c_row = np.stack([x, np.zeros_like(x), np.zeros_like(x)], 1)
    c_field = _lattice_points(400, 1.5, rng, exclude=lambda p: np.hypot(p[:, 1], p[:, 2]) < 1.5)
    c = np.concatenate([c_row, c_field]); r = np.concatenate([np.full(len(x), 0.3), rng.uniform(0.1, 0.6, 400)])
    return _scene(c, r, rng)


def overlap_lattice(seed=0):
    """14^3 spheres of radius 0.3 .. 0.4 every 0.5: neighbours overlap, and a line across the block has ~20 with disc >= 0"""
    rng = np.random.default_rng(5000 + seed)
    g = (np.arange(14) - 6.5) * 0.5
    c = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + rng.uniform(-0.01, 0.01, (14 ** 3, 3))
    return _scene(c, rng.uniform(0.3, 0.4, len(c)), rng)


def big_not_f32(seed=0):
    """a ground of radius 1000.1 at y = -1000.1 and a second large sphere, neither representable in f32 (the f32 fast path of
    the large spheres is off: every lane takes the f64 routine), under 300 small f32 spheres"""
    rng = np.random.default_rng(6000 + seed)
    small = f32_scene(dict(center=_lattice_points(300, 1.5, rng) + [0.0, 8.0, 0.0], radius=rng.uniform(0.1, 0.6, 300)))
    c = np.concatenate([small["center"], [[0.0, -1000.1, 0.0], [20.1, 12.7, -30.3]]])
    r = np.concatenate([small["radius"], [1000.1, 12.3]])
    arrays = _scene(c, r, rng, exact=True)
    return {**arrays, "mat_albedo": f32(arrays["mat_albedo"]), "mat_param": f32(arrays["mat_param"])}


def random_scene(capi, half_extent, seed=1):
    return f32_scene(capi.random_scene(seed, half_extent))


# name -> (builder(capi), {backend: arm}): the arm plan_scan must pick for SCAN_AUTO, SCAN_FP32 and SCAN_TENSOR (None: refused)
def _arms(auto, fp32, tensor):
    return {SCAN_AUTO: auto, SCAN_FP32: fp32, SCAN_TENSOR: tensor}


TENSOR_SMEM, TENSOR_WIDE = _arms("Tensor", "Smem", "Tensor"), _arms("Tensor", "Wide", "Tensor")
SCENES = {
    # compact, R ~ 10: words of 32 (the FP32 filter), chunks of 64 (the tensor image), and the 1024-sphere FP32 segment
    **{f"compact-{n}": (lambda capi, n=n: compact(n), TENSOR_SMEM) for n in (1, 63, 64, 65, 127, 129, 1031)},
    "compact-1057": (lambda capi: compact(1057), TENSOR_SMEM),        # a second FP32 segment; one sphere in the partial word
    "compact-1100": (lambda capi: compact(1100), TENSOR_SMEM),        # a second FP32 segment; three records in the partial word
    "compact-3040": (lambda capi: compact(3040), TENSOR_SMEM),        # np 3040: the largest FP32 table of a 256-thread CTA
    "compact-3072": (lambda capi: compact(3072), TENSOR_WIDE),        # np 3072: the first that needs the wide CTA
    "compact-3137": (lambda capi: compact(3137), TENSOR_WIDE),        # npad 3200 with 63 padding columns past `small`
    "compact-3200": (lambda capi: compact(3200), TENSOR_WIDE),        # npad 3200: the largest tensor image that fits
    "compact-3201": (lambda capi: compact(3201), _arms("Wide", "Wide", None)),       # npad 3264: fails the smem rule only
    "compact-13472": (lambda capi: compact(13472), _arms("Wide", "Wide", None)),     # np 13472: the largest wide table
    "compact-13504": (lambda capi: compact(13504), _arms("Global", "Global", None)),  # np 13504: the table stays in global memory
    "row-r0.2": (lambda capi: row(0.2), _arms("Smem", "Smem", None)),  # slack 0.155 > mean r^2 0.04: fails the slack rule only
    "row-r0.4": (lambda capi: row(0.4), TENSOR_SMEM),                  # slack 0.156 < mean r^2 0.16
    "ball-R130": (lambda capi: sparse_ball(130.0), _arms("Smem", "Smem", None)),     # 4 R^2 > 60000: fails d_fits only
    "ball-R121": (lambda capi: sparse_ball(121.0), TENSOR_SMEM),       # Rp = 128, ns mod 64 = 25: padding past `small`
    "field-row": (lambda capi: field_row(), TENSOR_SMEM),             # candidate overflow
    "overlap-lattice": (lambda capi: overlap_lattice(), TENSOR_SMEM),  # candidate overflow
    "big-not-f32": (lambda capi: big_not_f32(), TENSOR_SMEM),
    "final": (lambda capi: random_scene(capi, 11), TENSOR_SMEM),
    "final-h27": (lambda capi: random_scene(capi, 27), TENSOR_SMEM),
    "final-h28": (lambda capi: random_scene(capi, 28), _arms("Wide", "Wide", None)),
    "final-h63": (lambda capi: random_scene(capi, 63), _arms("Global", "Global", None)),
}


@lru_cache(maxsize=None)
def _built(name, capi):
    return SCENES[name][0](capi)


def build(name, capi):
    """the scene's arrays (built once per process; callers must not modify them)"""
    return _built(name, capi)


# ------------------------------------------------------------------------------------------------ rays
def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def per_sphere_rays(arrays, seed=0):
    """two rays per small sphere: one from its centre in a random direction (it must leave through its own wall) and one
    from 1.5 .. 3 |r| outside it, aimed at its centre"""
    rng = np.random.default_rng(7000 + seed)
    k = scene_info(arrays)["small"]
    c, r = arrays["center"][k], np.abs(arrays["radius"][k])
    u = _unit(rng.normal(size=(len(k), 3))); v = _unit(rng.normal(size=(len(k), 3)))
    o_in, d_in = c, u * rng.uniform(0.5, 2.0, (len(k), 1))
    o_out = c + v * (r * rng.uniform(1.5, 3.0, len(k)))[:, None]
    d_out = -v * rng.uniform(0.5, 2.0, (len(k), 1))
    return np.concatenate([o_in, o_out]), np.concatenate([d_in, d_out])


def framing(arrays):
    """(spheres of interest, their middle, an extent around it, a camera eye that sees them): the view of mixed_rays' camera rays"""
    info = scene_info(arrays)
    k_all = info["small"] if info["ns"] else np.arange(len(arrays["radius"]))
    cs, r = arrays["center"][k_all], np.abs(arrays["radius"][k_all])
    mid = cs.mean(0)
    ext = float(np.percentile(np.linalg.norm(cs - mid, axis=1), 90)) + r.max() + 1.0
    return k_all, mid, ext, mid + 1.4 * ext * _unit(np.array([0.8, 0.35, 0.5]))


def mixed_rays(arrays, n=4000, seed=0):
    """camera rays, rays leaving sphere surfaces, origins 30 .. 2000 away aimed at a sphere, short directions, and lines that
    miss the bounding sphere of the small spheres"""
    rng = np.random.default_rng(8000 + seed)
    info = scene_info(arrays)
    c, r = arrays["center"], np.abs(arrays["radius"])
    k_all, mid, ext, eye = framing(arrays)
    n_cam, n_sec, n_far, n_short, n_miss = (int(n * f) for f in (0.3, 0.3, 0.2, 0.1, 0.1))
    o_cam = eye + 0.05 * rng.normal(size=(n_cam, 3))
    d_cam = mid + ext * _unit(rng.normal(size=(n_cam, 3))) * rng.uniform(0, 1, (n_cam, 1)) ** (1 / 3) - o_cam
    k = rng.choice(k_all, n_sec + n_short)
    o_sec = c[k] + _unit(rng.normal(size=(len(k), 3))) * (r[k] * 1.05)[:, None]
    d_sec = rng.normal(size=(len(k), 3)) * rng.uniform(0.05, 2.0, (len(k), 1))
    d_sec[n_sec:] *= 1e-3                                                # short directions: t scales, the hit does not
    k = rng.choice(k_all, n_far)
    target = c[k] + _unit(rng.normal(size=(n_far, 3))) * (r[k] * rng.uniform(0, 0.6, n_far))[:, None]
    u = _unit(rng.normal(size=(n_far, 3)))
    o_far = target + u * 10 ** rng.uniform(1.5, 3.3, (n_far, 1)); d_far = -u * rng.uniform(0.3, 3.0, (n_far, 1))
    u = _unit(rng.normal(size=(n_miss, 3))); w = _unit(np.cross(u, rng.normal(size=(n_miss, 3))))
    o_miss = w * (info["R"] * rng.uniform(1.2, 3.0, (n_miss, 1))) + u * rng.uniform(0, 2 * info["R"], (n_miss, 1))
    d_miss = -u * rng.uniform(0.5, 2.0, (n_miss, 1))
    return np.concatenate([o_cam, o_sec, o_far, o_miss]), np.concatenate([d_cam, d_sec, d_far, d_miss])


def row_rays(x0, x1, n=1000, seed=0):
    """rays along the x axis into a row of spheres on it (from either end, up to 0.15 off the axis, nearly parallel to it)"""
    rng = np.random.default_rng(9000 + seed)
    side = rng.choice([-1.0, 1.0], n)
    o = np.stack([np.where(side < 0, x1 + rng.uniform(1, 3, n), x0 - rng.uniform(1, 3, n)), rng.uniform(-0.15, 0.15, n),
                  rng.uniform(-0.15, 0.15, n)], 1)
    d = np.stack([-side, rng.normal(0, 2e-3, n), rng.normal(0, 2e-3, n)], 1) * rng.uniform(0.5, 2.0, (n, 1))
    return o, d


def f32(a):
    return np.asarray(a, np.float32).astype(np.float64)


# ------------------------------------------------------------------------------------------------ silhouette rays
# The bands in which a filter can drop a hit, as designed (DESIGN.md §1.1, §1.2), in units of the discriminant of a unit
# direction (r^2 - dist(centre, line)^2).  Stated here rather than read from the sources, so that a changed slack cannot
# move the bands the tests demand rays in.
FP32_SLACK = 96 * 2.0 ** -24                    # RT_FILTER_SLACK: per unit of |c|^2 + r^2 + R^2
TENSOR_SLACK = 1.5625e-5                        # tensor_image: per unit of R^2
SIGMA_PER_LEN = 16 * 2.0 ** -24                 # sigma = this x max |r| x |o|_1 (rtiow_scene_upload, line_gate)
SIL_DELTA = (-3e-2, -1e-2, -3e-3, -1e-3, -3e-4, -1e-4, -3e-5, -1e-5, 0.0, 1e-5, 3e-5, 1e-4, 3e-4, 1e-3)
SIL_BAND = (0.01, 0.1, 0.5, 0.9)                # lines whose discriminant is this fraction of each filter's band
SIL_BACK = (0.0, 10.0, 100.0, 1000.0, 3000.0)   # origin distance behind the line's closest point (0: 3 |r|)
SIL_DLEN = (1e-3, 1.0, 30.0)


def _perp(u, rng):
    """a random unit vector perpendicular to each row of u"""
    return _unit(np.cross(u, rng.normal(size=u.shape)))


def _band_deltas(info, c, r):
    """per sphere, the deltas at which r^2 - (r (1 + delta))^2 is each SIL_BAND fraction of the tensor and the FP32 band"""
    tensor = TENSOR_SLACK * info["R"] ** 2
    fp32 = FP32_SLACK * ((c * c).sum(1) + r * r + info["R"] ** 2)
    disc = np.concatenate([np.multiply.outer(tensor * np.ones_like(r), SIL_BAND), np.multiply.outer(fp32, SIL_BAND)], 1)
    return np.sqrt(np.clip(1.0 - disc / (r * r)[:, None], 0.0, None)) - 1.0


def silhouette_rays(arrays, n_spheres=40, seed=0):
    """rays whose line passes within a hair of a small sphere's silhouette, where a filter's rounding decides:
      * per sampled sphere, lines |r| (1 + delta) from its centre for every SIL_DELTA and for the deltas that put the
        discriminant at SIL_BAND fractions of each filter's band, origins SIL_BACK behind the closest point, |d| in SIL_DLEN;
      * the same at the outermost spheres, on the side where they touch the bounding R-sphere (lines that graze it: the
        live gate and the R^2 margin);
      * axis-aligned directions (exact zeros), origins at the coordinate origin, and origins on sphere surfaces, aimed past a
        sphere's silhouette or in random directions.
    -> (o, d, target): f32-rounded rays and, per ray, the list index of the sphere whose silhouette it was built on."""
    rng = np.random.default_rng(10000 + seed)
    info = scene_info(arrays)
    ks = info["small"]
    C, Rad = np.asarray(arrays["center"], float), np.abs(np.asarray(arrays["radius"], float))
    sample = rng.choice(ks, n_spheres, replace=len(ks) < n_spheres)       # a scene of few spheres: each one several times
    reach = np.linalg.norm(C[ks], axis=1) + Rad[ks]
    outer = ks[np.argsort(-reach, kind="stable")[:8]]
    os_, ds, ts = [], [], []

    def add(o, d, k):
        os_.append(o); ds.append(d); ts.append(k)

    def grid(k, radial):
        """every (delta, back, |d|) for the spheres k; radial: the closest point lies on the far side from the coordinate origin"""
        deltas = np.concatenate([np.tile(SIL_DELTA, (len(k), 1)), _band_deltas(info, C[k], Rad[k])], 1)
        nd = deltas.shape[1]
        kk = np.repeat(k, nd * len(SIL_BACK) * len(SIL_DLEN))
        delta = np.repeat(deltas.reshape(-1), len(SIL_BACK) * len(SIL_DLEN))
        back = np.tile(np.repeat(SIL_BACK, len(SIL_DLEN)), len(k) * nd)
        dlen = np.tile(SIL_DLEN, len(k) * nd * len(SIL_BACK))
        c, r = C[kk], Rad[kk]
        if radial:
            w = np.where(np.linalg.norm(c, axis=1)[:, None] > 0, c, rng.normal(size=c.shape))
            w = _unit(w); u = _perp(w, rng)
        else:
            u = _unit(rng.normal(size=c.shape)); w = _perp(u, rng)
        back = np.where(back == 0.0, 3.0 * r, back)
        q = c + w * (r * (1.0 + delta))[:, None]
        add(q - u * back[:, None], u * dlen[:, None], kk)

    grid(sample, False)
    grid(outer, True)
    # axis-aligned: direction +-e_i, the line offset from the centre along e_j
    for i in range(3):
        for s in (-1.0, 1.0):
            kk = np.repeat(sample[:20], len(SIL_DELTA) * 2)
            delta = np.tile(SIL_DELTA, len(sample[:20]) * 2)
            back = np.tile(np.repeat([0.0, 100.0], len(SIL_DELTA)), len(sample[:20]))
            c, r = C[kk], Rad[kk]
            back = np.where(back == 0.0, 3.0 * r, back)
            e_i, e_j = np.eye(3)[i], np.eye(3)[(i + 1) % 3]
            add(c + e_j * (r * (1.0 + delta))[:, None] - s * e_i * back[:, None], np.tile(s * e_i, (len(kk), 1)), kk)
    # origins at the coordinate origin, aimed past a silhouette, and along the axes
    kk = np.repeat(sample, len(SIL_DELTA))
    delta = np.tile(SIL_DELTA, len(sample))
    c, r = C[kk], Rad[kk]
    w = _perp(np.where(np.linalg.norm(c, axis=1)[:, None] > 0, c, rng.normal(size=c.shape)), rng)
    add(np.zeros_like(c), c + w * (r * (1.0 + delta))[:, None], kk)
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    add(np.zeros((12, 3)), np.concatenate([axes, 1e-3 * axes]), np.full(12, sample[0]))
    # origins on a sphere's surface: aimed past another sphere's silhouette, and in random directions
    k1, k2 = np.repeat(sample, len(SIL_DELTA)), rng.choice(ks, len(sample) * len(SIL_DELTA))
    o = C[k1] + _unit(rng.normal(size=(len(k1), 3))) * Rad[k1][:, None]
    w = _perp(C[k2] - o, rng)
    add(o, C[k2] + w * (Rad[k2] * (1.0 + np.tile(SIL_DELTA, len(sample))))[:, None] - o, k2)
    add(o, _unit(rng.normal(size=o.shape)) * rng.uniform(0.5, 2.0, (len(o), 1)), k1)
    o, d, t = np.concatenate(os_), np.concatenate(ds), np.concatenate(ts)
    keep = np.linalg.norm(d, axis=1) > 0                # (a sphere centred on the coordinate origin has no silhouette point there)
    return f32(o[keep]), f32(d[keep]), t[keep]


def silhouette_bands(arrays, o, d, target):
    """per ray, the f64 discriminant of its target sphere for the f32-rounded inputs and the unit direction, r^2 - dist^2, and
    the two bands in which a filter may err: the tensor slack, and the FP32 slack + the ray's sigma (its origin's foot point)
    -> dict(disc, tensor, fp32)"""
    info = scene_info(arrays)
    c = np.asarray(arrays["center"], float)[target]; r = np.asarray(arrays["radius"], float)[target]
    u = d / np.linalg.norm(d, axis=1, keepdims=True)
    x = np.cross(o - c, u)                              # dist(centre, line) without the cancellation of |oc|^2 - hb^2
    disc = r * r - (x * x).sum(1)
    rmax = max(float(np.abs(np.asarray(arrays["radius"], float)[info["small"]]).max()), 1e-3)
    sigma = SIGMA_PER_LEN * rmax * np.abs(o).sum(1)
    return dict(disc=disc, tensor=np.full(len(o), TENSOR_SLACK * info["R"] ** 2),
                fp32=FP32_SLACK * ((c * c).sum(1) + r * r + info["R"] ** 2) + sigma)


def band_coverage(arrays, o, d, target):
    """how many rays fall inside each band (0 < disc <= band), and inside its first 1 %"""
    b = silhouette_bands(arrays, o, d, target)
    pos = b["disc"] > 0
    return {f"{k}{tag}": int((pos & (b["disc"] <= f * b[k])).sum()) for k in ("tensor", "fp32") for tag, f in (("", 1.0), ("_1%", 0.01))}


def assert_band_coverage(arrays, o, d, target, need=300, need_edge=50):
    """a weak ray set fails here instead of passing vacuously"""
    cov = band_coverage(arrays, o, d, target)
    assert cov["tensor"] >= need and cov["fp32"] >= need, cov
    assert cov["tensor_1%"] >= need_edge and cov["fp32_1%"] >= need_edge, cov
    return cov


# rays along the row of spheres that overflows the candidate lists, for the scenes that have one
EXTRA_RAYS = {"field-row": lambda: row_rays(-10.0, 10.0), "row-r0.2": lambda: row_rays(0.0, 99.5),
              "row-r0.4": lambda: row_rays(0.0, 99.5)}


def rays(name, arrays, seed=0, n_mixed=4000):
    """the per-sphere rays, the mixed set and the scene's extra rays, f32-rounded"""
    parts = [per_sphere_rays(arrays, seed), mixed_rays(arrays, n_mixed, seed)]
    if name in EXTRA_RAYS:
        parts.append(EXTRA_RAYS[name]())
    return f32(np.concatenate([p[0] for p in parts])), f32(np.concatenate([p[1] for p in parts]))


# ------------------------------------------------------------------------------------------------ f64 reference
def _line_terms(c, r2, o, d):
    """a = |d|^2, hb = (c - o).d and disc = hb^2 - a (|o - c|^2 - r^2) for every (ray, sphere) pair, through matrix products
    (|o - c|^2 expanded: in f64 its cancellation costs ~1e-16 |o|^2, far below the knife-edge margins used here)"""
    a = (d * d).sum(1)[:, None]
    hb = d @ c.T - (d * o).sum(1)[:, None]
    cc = ((o * o).sum(1)[:, None] - 2.0 * (o @ c.T)) + ((c * c).sum(1) - r2)[None]
    return a, hb, hb * hb - a * cc


def robust_closest(arrays, o, d, t_min=1e-4, chunk_pairs=1 << 22):
    """closest hit of every ray over all spheres in f64 (sphere.rs:16-34, mod.rs:56-69: ties go to the later list index)
    -> dict(index, t, t2, robust).  t2 is the second-smallest root any sphere offers (each sphere offers the root the reference
    would accept).  A hit is robust when its sphere is not grazed (not_grazing), the next sphere's root lies more than
    1e-5 (|o| + R) further along the ray (as a length), and t is not within 1e-5 of t_min."""
    c = np.asarray(arrays["center"], float); r = np.asarray(arrays["radius"], float)
    n, m = len(o), len(r)
    idx = np.full(n, -1); t1 = np.full(n, np.inf); t2 = np.full(n, np.inf)
    step = max(1, chunk_pairs // max(m, 1))
    for s in range(0, n, step):
        a, hb, disc = _line_terms(c, r * r, o[s:s + step], d[s:s + step])
        sq = np.sqrt(np.maximum(disc, 0.0))
        near = (hb - sq) / a
        root = np.where(near >= t_min, near, (hb + sq) / a)
        root[(disc < 0) | (root < t_min)] = np.inf
        last = m - 1 - np.argmin(root[:, ::-1], axis=1)                 # the later index among equal roots
        two = np.partition(root, 1, axis=1)[:, :2] if m > 1 else np.concatenate([root, np.full((len(root), 1), np.inf)], 1)
        t1[s:s + step], t2[s:s + step] = two[:, 0], two[:, 1]
        idx[s:s + step] = np.where(np.isfinite(two[:, 0]), last, -1)
    hi = np.maximum(idx, 0)
    dl = np.linalg.norm(d, axis=1)
    R = scene_info(arrays)["R"]
    with np.errstate(invalid="ignore"):                                 # inf - inf on rays that hit nothing
        gap = (t2 - t1) * dl > 1e-5 * (np.linalg.norm(o, axis=1) + R)
    robust = (idx >= 0) & not_grazing(c[hi], r[hi], o, d) & gap & (np.abs(t1 - t_min) > 1e-5)
    return dict(index=idx, t=t1, t2=t2, robust=robust)


def line_survivors(arrays, o, d):
    """per ray, how many small spheres its LINE meets (disc >= 0 in f64): a lower bound on the filter's survivors"""
    k = scene_info(arrays)["small"]
    c, r = np.asarray(arrays["center"], float)[k], np.asarray(arrays["radius"], float)[k]
    out = np.zeros(len(o), int)
    step = max(1, (1 << 22) // max(len(k), 1))
    for s in range(0, len(o), step):
        out[s:s + step] = (_line_terms(c, r * r, o[s:s + step], d[s:s + step])[2] >= 0).sum(1)
    return out
