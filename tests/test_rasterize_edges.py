"""The label rasteriser (`b2_rasterize_polygons`, `ops.rasterize_polygons`) where scanline and edge-walk code goes wrong.

* An exact rational restatement of GDAL's pixel-centre rule (`_exact_fill`), written in closed form rather than as the
  oracle's scanline loop, on dyadic lattice polygons: every vertex a multiple of 1/4, every non-horizontal edge with |dy| a
  power of two, so that every double operation of the crossing formula is exact and the oracle, the kernel and the
  reference must agree bit for bit, ties on pixel centres and pixel corners included.
* Kernel against the oracle, bit for bit, with and without ALL_TOUCHED: GDAL's 0.01 shortcuts, edges one ulp off integers
  and half-integers, clipping on every side and corner, vertices at +-1e9 and +-1e15, 1x1 to 4096x4096 rasters, 5 000
  overlapping features, features with no scanline on the raster anywhere in the burn order, and the drop-in
  `create_label_array_for_tile` on GeoJSON layers digitised on the tile's own grid.
* Layer-scale inputs: one very detailed feature off the tile's rows next to thousands of small ones (the scanline
  workspace follows the crossings), a feature a trillion pixels away, non-finite vertices, out-of-range burn values and
  rasters of 2^31 pixels or more.
"""
import json
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import rasterize as orr


# ------------------------------------------------------------------------------------------------ exact reference
def _rings_of(rings):
    """The rings GDAL's fill walks: at least two vertices given, the duplicated closing vertex dropped."""
    out = []
    for r in rings:
        r = np.asarray(r, dtype=np.float64).reshape(-1, 2)
        if len(r) < 2:
            continue
        out.append(r[:-1] if r[0, 0] == r[-1, 0] and r[0, 1] == r[-1, 1] else r)
    return out


def _exact_fill(features, H, W, background=255):
    """GDAL's pixel-centre burn in closed form, in rational arithmetic.  Pixel (x, y), centre c = (x + 1/2, y + 1/2), is
    burnt by a feature iff y is one of its visited rows [max(trunc(min y), 0), min(trunc(max y), H - 1)] and
    (a) an odd number of its non-horizontal edges have y_lo <= c_y < y_hi and cross y = c_y at an X < c_x, or
    (b) one of its horizontal edges lies on y = c_y, runs right to left and has cur.x < c_x <= prev.x.
    The last feature to burn a pixel wins."""
    out = np.full((H, W), background, np.uint8)
    cx = [Fraction(2 * x + 1, 2) for x in range(W)]
    for rings, value in features:
        rings = _rings_of(rings)
        if not rings:
            continue
        edges = [tuple(Fraction(float(v)) for v in (r[i - 1, 0], r[i - 1, 1], r[i, 0], r[i, 1]))
                 for r in rings for i in range(len(r))]
        ys = [e[1] for e in edges]
        for y in range(max(math.trunc(min(ys)), 0), min(math.trunc(max(ys)), H - 1) + 1):
            cy = Fraction(2 * y + 1, 2)
            xs, burn = [], np.zeros(W, bool)
            for px, py, qx, qy in edges:
                if py != qy:
                    if min(py, qy) <= cy < max(py, qy):
                        xs.append(px + (cy - py) * (qx - px) / (qy - py))
                elif py == cy and px > qx:
                    burn |= np.array([qx < c <= px for c in cx])
            burn |= np.array([sum(X < c for X in xs) % 2 == 1 for c in cx])
            out[y, burn] = value
    return out


# ------------------------------------------------------------------------------------------------ lattice layers
_POW2 = [0.25 * 2 ** k for k in range(9)]             # 1/4 .. 64


def _lattice_ring(rng, n, start, dmax=16.0, span=10.0):
    """A random closed walk of n steps on the 1/4 lattice: every non-horizontal step has |dy| a power of two (paired +-d
    so that it closes), the closing step included; often self-intersecting (the even-odd rule applies)."""
    pows = [d for d in _POW2 if d <= dmax]
    dys = []
    while len(dys) + 2 <= n:
        if rng.random() < 0.25:
            dys.append(0.0)
        else:
            d = float(rng.choice(pows))
            dys += [d, -d]
    dys += [0.0] * (n - len(dys))
    dys = np.array(dys)[rng.permutation(n)]
    dxs = rng.integers(-int(4 * span), int(4 * span) + 1, n) / 4.0
    dxs[-1] = -dxs[:-1].sum()
    v = np.asarray(start, np.float64) + np.cumsum(np.stack([dxs, dys], 1), axis=0)
    return np.vstack([v[-1:], v[:-1]])                   # starts at `start`; the last step returns to it


def _hand_shapes():
    """Lattice shapes with every |dy| a power of two: (name, rings)."""
    A = lambda *p: np.array(p, np.float64)
    return [
        ("square", [A((2, 2), (10, 2), (10, 10), (2, 10), (2, 2))]),
        ("triangle on centres", [A((3.5, 1.5), (11.5, 1.5), (7.5, 5.5), (3.5, 1.5))]),
        ("diamond", [A((8, 0.5), (12, 4.5), (8, 8.5), (4, 4.5))]),
        ("U (concave)", [A((1, 1), (3, 1), (3, 5), (7, 5), (7, 1), (9, 1), (9, 9), (1, 9), (1, 1))]),
        ("shell with hole", [A((1, 1), (15, 1), (15, 17), (1, 17), (1, 1)), A((5, 5), (5, 9), (9, 9), (9, 5), (5, 5))]),
        ("hole on the shell's edge", [A((1, 1), (13, 1), (13, 9), (1, 9), (1, 1)), A((1, 3), (5, 3), (5, 5), (1, 5), (1, 3))]),
        ("hole touching at a vertex", [A((1, 1), (13, 1), (13, 9), (1, 9), (1, 1)), A((7, 1), (9, 3), (7, 5), (5, 3), (7, 1))]),
        ("bow-tie", [A((2, 2), (10, 10), (10, 2), (2, 10), (2, 2))]),
        ("overlapping parts", [A((2, 2), (10, 2), (10, 10), (2, 10), (2, 2)), A((6, 6), (14, 6), (14, 14), (6, 14), (6, 6))]),
        ("edges on centre lines, clockwise", [A((2, 2.5), (12, 2.5), (12, 10.5), (2, 10.5), (2, 2.5))]),
        ("edges on centre lines, anticlockwise", [A((2, 2.5), (2, 10.5), (12, 10.5), (12, 2.5), (2, 2.5))]),
        ("half-pixel box", [A((1.5, 1.5), (9.5, 1.5), (9.5, 3.5), (5.5, 3.5), (5.5, 5.5), (1.5, 5.5))]),
        ("2-vertex ring", [A((3, 3), (9, 7))]),
        ("closed 2-vertex ring", [A((3, 3.5), (9, 7.5), (3, 3.5))]),
        ("3-vertex ring", [A((2, 1), (10, 5), (4, 9))]),
        ("unclosed with repeated vertices", [A((2, 2), (2, 2), (10, 2), (10, 10), (10, 10), (2, 10))]),
        ("one-vertex ring beside a square", [A((4, 4)), A((2, 2), (6, 2), (6, 6), (2, 6))]),
    ]


def _lattice_layers():
    """Seeded layers of lattice polygons: (name, features, (H, W))."""
    rng = np.random.default_rng(2024)
    shapes = _hand_shapes()
    layers = [("hand shapes %s" % name, [(rings, 7)], (16, 20)) for name, rings in shapes]
    for it, size in enumerate([(16, 16), (33, 20), (64, 64), (1, 9), (9, 1), (24, 40), (64, 48), (5, 64)]):
        H, W = size
        feats = []
        for f in range(int(rng.integers(6, 18))):
            q = lambda lo, hi: rng.integers(int(4 * lo), int(4 * hi) + 1) / 4.0
            off = np.array([q(-6, W), q(-6, H)])
            if f % 3 == 0:
                rings = [r + off for r in shapes[int(rng.integers(len(shapes)))][1]]
            else:
                rings = [_lattice_ring(rng, int(rng.integers(3, 11)), off, dmax=min(16.0, 2.0 ** int(np.log2(max(H, 2)))))
                         for _ in range(int(rng.integers(1, 3)))]
                if f % 4 == 1:                               # given closed (the first vertex repeated)
                    rings = [np.vstack([r, r[:1]]) for r in rings]
            feats.append((rings, int(rng.integers(0, 256))))
        layers.append(("random lattice %d" % it, feats, size))
    return layers


def _exact_inputs(features):
    """Every vertex on the 1/4 lattice and every non-horizontal fill edge with |dy| a power of two from 1/4 to 64."""
    for rings, _ in features:
        for r in _rings_of(rings):
            assert (r * 4 == np.round(r * 4)).all() and (np.abs(r) < 2 ** 20).all()
            dy = np.abs(r[:, 1] - np.roll(r[:, 1], 1))
            assert all(d == 0 or d in _POW2 for d in dy), dy
    return True


# ------------------------------------------------------------------------------------------------ oracle-only layers
def _star(rng, c, rx, ry, k):
    ang = np.sort(rng.random(k)) * 2 * np.pi
    rad = rng.uniform(0.3, 1.0, k)
    ring = np.stack([c[0] + rx * rad * np.cos(ang), c[1] + ry * rad * np.sin(ang)], 1)
    return np.vstack([ring, ring[:1]])


def _stars(rng, n, H, W, kmax=10):
    """n random star polygons over (and hanging off) an H x W raster, sized to each axis; values 0..255."""
    feats = []
    for f in range(n):
        c = rng.uniform(-0.1, 1.1, 2) * (W, H)
        rings = [_star(rng, c, max(0.6 * W * rng.random(), 0.7), max(0.6 * H * rng.random(), 0.7), int(rng.integers(3, kmax)))]
        if f % 3 == 0:
            rings.append((c + (rings[0] - c) * 0.4)[::-1].copy())
        feats.append((rings, int(rng.integers(0, 256))))
    return feats


def _shortcut_layers():
    """Edges just below / at / above GDAL's 0.01 near-axis-parallel shortcuts, inside one pixel column or row, and one ulp
    off an integer or a half-integer, each as one side of a polygon (single-feature layers on 24 x 24)."""
    layers = []
    up, dn = lambda v: np.nextafter(v, np.inf), lambda v: np.nextafter(v, -np.inf)
    for d in (0.0099, 0.00999999, 0.01, 0.0100001, 0.012, 0.015, 0.0199, 0.02, 0.021):
        for x0, ya, yb in ((6.0, 2.3, 19.7), (11.0, 20.6, 1.2)):
            p, q = (x0 - d / 2, ya), (x0 + d / 2, yb)
            for far in (21.3, 1.7):                            # the polygon on either side of the edge
                ring = np.array([p, q, (far, 0.5 * (ya + yb) + 1.1), p])
                layers.append(("near-vertical dx=%g x0=%g far=%g" % (d, x0, far), [([ring], 9)]))
                layers.append(("near-horizontal dy=%g y0=%g far=%g" % (d, x0, far), [([ring[:, ::-1].copy()], 9)]))
    for p, q in (((5.1, 2.2), (5.9, 20.6)), ((5.02, 20.6), (5.98, 2.2)), ((0.3, 3.7), (0.7, 22.1))):
        for ring in (np.array([p, q, (17.0, 12.3), p]), np.array([p, (17.0, 12.3), q, p])):
            layers.append(("inside one column", [([ring], 3)]))
            layers.append(("inside one row", [([ring[:, ::-1].copy()], 3)]))
    for a in (6.0, 5.5, 12.0, 0.0, 24.0, 0.5, 23.5):
        for f in (up, dn):
            b = f(a)
            rings = [np.array([(b, 2.5), (18.25, 2.5), (18.25, b), (b, 18.5), (b, 2.5)]),
                     np.array([(3.0, b), (20.0, 3.5), (f(a + 7.0), 21.0), (3.0, b)])]
            layers.append(("one ulp off %g" % a, [(rings[:1], 5), (rings[1:], 6)]))
            layers.append(("one ulp off %g, one feature" % a, [(rings, 4)]))
    return [(name, feats, (24, 24)) for name, feats in layers]


def _clip_layers():
    """Polygons over each side and corner, wholly outside, containing the raster, with vertices at +-1e9 / +-1e15 (edges
    kept axis-parallel or of moderate slope: how long GDAL's walk runs outside the raster is not under test), and a
    steep edge through the top and the bottom; on 20 x 30."""
    H, W = 20, 30
    R = lambda x0, y0, x1, y1: np.array([(x0, y0), (x1, y0), (x1, y1), (x0, y1), (x0, y0)], np.float64)
    T = lambda *p: np.array(p + (p[0],), np.float64)
    over = [R(-5.3, 4.2, 6.7, 11.9), R(23.6, 3.3, 36.1, 9.8), R(4.4, -7.2, 12.5, 5.5), R(7.7, 14.1, 19.2, 26.6),
            R(-3.3, -4.4, 5.5, 6.6), R(24.5, -2.5, 33.5, 5.5), R(-2.25, 15.75, 4.75, 23.25), R(26.2, 16.8, 31.9, 21.4),
            T((-4.1, 2.2), (8.3, 10.9), (-6.6, 17.3)), T((33.1, -3.2), (22.4, 9.9), (35.7, 24.8))]
    outside = [R(-9.0, 3.0, -1.0, 9.0), R(31.0, 3.0, 40.0, 9.0), R(3.0, -12.0, 9.0, -0.5), R(3.0, 20.0, 9.0, 29.0),
               R(-9.0, -9.0, -0.01, -0.01), R(30.0, 20.0, 31.0, 21.0), T((-1e9, 5.0), (-3.0, 9.0), (-7.0, 1e9)),
               R(-1e15, -1e15, 1e15, -0.25)]
    big, huge = 1e9, 1e15
    far = [R(-huge, -huge, huge, huge), R(-big, -big, big, big), R(-2.0, -1.0, W + 2.0, H + 1.0),
           R(-huge, 3.5, 7.25, 9.75), R(-huge, 3.5, 7.25, 9.75)[::-1].copy(), R(22.25, 12.5, huge, 16.5),
           R(4.3, -huge, 5.6, huge), R(11.5, -big, 12.5, big), R(-big, 17.2, big, 17.8),
           T((2.2, 3.1), (big, big + 1.3), (big - 7.0, big)), T((-big, -big), (12.3, 4.1), (-big, 2.7)),
           T((-huge, -huge), (12.3, 4.1), (-huge, 2.7)), T((27.7, 18.2), (huge, huge), (-huge, huge)),
           T((-huge, 5.3), (huge, 7.7), (huge, 11.1)), T((5.5, 10.5), (huge, 10.5), (huge, huge))]
    steep = [T((10.3, -50.0), (12.9, 70.0), (20.1, 10.2)), T((17.6, 44.0), (16.1, -31.0), (3.3, 8.8))]
    layers = []
    for name, group in (("over the edge", over), ("outside", outside), ("far vertices", far), ("steep", steep)):
        for i, ring in enumerate(group):
            layers.append(("%s %d" % (name, i), [([ring], 11)], (H, W)))
        layers.append(("%s, all" % name, [([r], 20 + i) for i, r in enumerate(group)], (H, W)))
    return layers


def _shape_layers():
    """Raster shapes 1x1, 1xN, Nx1, 3x2000, 2000x3."""
    rng = np.random.default_rng(77)
    layers = []
    for H, W in ((1, 1), (1, 37), (41, 1), (3, 2000), (2000, 3), (2, 2)):
        feats = _stars(rng, 12, H, W)
        feats.append(([np.array([(0.2, 0.3), (W - 0.1, 0.45), (W - 0.3, H - 0.2), (0.1, H - 0.4), (0.2, 0.3)])], 201))
        layers.append(("%dx%d" % (H, W), feats, (H, W)))
    return layers


def _zero_row_feature(kind, H, W):
    return {"above": [np.array([(2.0, -7.0), (9.0, -6.5), (5.0, -2.0), (2.0, -7.0)])],
            "below": [np.array([(2.0, H + 1.0), (9.0, H + 3.5), (5.0, H + 9.0), (2.0, H + 1.0)])],
            "empty": [],
            "one vertex": [np.array([(4.0, 4.0)])],
            "far below": [np.array([(1.0, 1e12), (30.0, 1e12 + 3.0), (12.0, 1e12 + 9.0), (1.0, 1e12)])]}[kind]


def _order_layers():
    """Burn order: features with no scanline on the raster first, last and between overlapping ones (equal job offsets);
    a layer ending in an empty feature."""
    H, W = 32, 32
    rng = np.random.default_rng(8)
    body = _stars(rng, 6, H, W)
    kinds = ["above", "below", "empty", "one vertex", "far below"]
    layers = []
    for k in kinds:
        z = lambda: (_zero_row_feature(k, H, W), 99)
        feats = [z(), body[0], z(), z(), body[1], body[2], z(), body[3], z(), z(), z(), body[4], body[5], z()]
        layers.append(("zero rows: %s" % k, feats, (H, W)))
    layers.append(("ends empty", body + [([], 3)], (H, W)))
    layers.append(("all zero rows", [(_zero_row_feature(k, H, W), 5) for k in kinds], (H, W)))
    return layers


def _overlap_layer():
    """5 000 small overlapping features whose values cycle through 0..255, on 96 x 96."""
    rng = np.random.default_rng(5000)
    feats = []
    for f in range(5000):
        c = rng.uniform(-2, 98, 2)
        feats.append(([_star(rng, c, rng.uniform(0.8, 5.0), rng.uniform(0.8, 5.0), int(rng.integers(3, 7)))], f % 256))
    return feats


def _layer_scale(rng=None):
    """A 512 x 512 tile: 2 000 small features on the tile, one feature of 200 000 vertices off the tile's rows (a coastline
    elsewhere in the file), one of 4 096 vertices spanning the tile."""
    rng = np.random.default_rng(512) if rng is None else rng
    feats = []
    for f in range(2000):
        c = rng.uniform(0, 512, 2)
        feats.append(([_star(rng, c, rng.uniform(1, 7), rng.uniform(1, 7), int(rng.integers(4, 11)))], int(rng.integers(0, 10))))
    coast = _star(rng, (256.0, -9000.0), 3000.0, 3000.0, 200_000)
    coast[:, 1] = np.minimum(coast[:, 1], -600.0)
    feats.insert(700, ([coast], 42))
    feats.insert(1500, ([_star(rng, (256.0, 256.0), 300.0, 300.0, 4096)], 43))
    return feats


# ------------------------------------------------------------------------------------------------ CPU
def test_exact_reference_agrees_with_the_oracle():
    """oracle.rasterize(all_touched=False) is GDAL's centre rule, ties included, on exact inputs."""
    layers = _lattice_layers()
    assert len(layers) >= 20
    for name, feats, (H, W) in layers:
        assert _exact_inputs(feats), name
        want = _exact_fill(feats, H, W, 255)
        got = orr.rasterize(feats, (H, W), 255, all_touched=False)
        assert np.array_equal(got, want), (name, np.argwhere(got != want)[:5].tolist())
    # the shapes burn what they should: a sanity check of the restatement itself on three hand cases
    sq = [([np.array([(2.0, 2.0), (6.0, 2.0), (6.0, 5.0), (2.0, 5.0)])], 1)]
    assert (_exact_fill(sq, 8, 8, 0) == 1).sum() == 12 and (_exact_fill(sq, 8, 8, 0)[2:5, 2:6] == 1).all()
    bow = [([np.array([(0.0, 0.0), (4.0, 4.0), (4.0, 0.0), (0.0, 4.0)])], 1)]
    assert _exact_fill(bow, 4, 4, 0).tolist() == [[1, 0, 0, 0], [1, 1, 0, 1], [1, 1, 0, 1], [1, 0, 0, 0]]   # ties at 3.5, 1.5
    centre = [([np.array([(1.0, 1.5), (1.0, 3.5), (3.0, 3.5), (3.0, 1.5)])], 1)]       # centre-line edge right to left
    assert _exact_fill(centre, 5, 5, 0)[1:4, 1:3].tolist() == [[1, 1], [1, 1], [0, 0]]


def _crossings(L, H):
    """What the kernel counts per job: non-horizontal fill edges of the job's feature with y_lo <= row + 0.5 < y_hi."""
    want = np.zeros(L.n_jobs, np.int64)
    for f in range(len(L.values)):
        j0, j1 = int(L.job_off[f]), int(L.job_off[f + 1])
        if j1 == j0:
            continue
        e = L.fill[L.fill_off[f]:L.fill_off[f + 1]]
        ylo, yhi = np.minimum(e[:, 1], e[:, 3]), np.maximum(e[:, 1], e[:, 3])
        cy = L.miny[f] + np.arange(j1 - j0)[:, None] + 0.5
        want[j0:j1] = ((ylo <= cy) & (cy < yhi) & (ylo != yhi)).sum(axis=1)
    return want


def test_host_workspace_bound_covers_every_crossing():
    """rasterize_layout's per-job room is at least the crossings the kernel's rule finds, on every layer of this file;
    features without scanlines get none, and a detailed feature off the tile costs the workspace nothing."""
    from dl_image_segmentation_b200 import ops
    layers = [(n, f, s) for n, f, s in _lattice_layers() + _shortcut_layers() + _clip_layers() + _shape_layers()
              + _order_layers()]
    layers += [("5000 overlapping", _overlap_layer(), (96, 96)), ("layer scale", _layer_scale(), (512, 512))]
    for name, feats, (H, W) in layers:
        for at in (True, False):
            L = ops.rasterize_layout(feats, (H, W), at)
            room = np.diff(L.job_ints_off.astype(np.int64))
            assert L.job_ints_off[0] == 0 and (room >= 0).all()
            assert (room >= _crossings(L, H)).all(), name
            rows = np.diff(L.job_off.astype(np.int64))
            assert ((L.miny >= 0) & (L.miny < H)).all() and (rows <= H).all(), name
    L = ops.rasterize_layout(_layer_scale(), 512)
    assert L.job_off[701] == L.job_off[700]                  # the 200 000-vertex feature has no rows on the tile
    assert int(L.job_ints_off[-1]) * 4 < (4 << 20), int(L.job_ints_off[-1])


def test_host_layout_refuses_bad_vertices_and_values():
    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    ok = np.array([(1.0, 1.0), (6.0, 1.5), (3.0, 5.0), (1.0, 1.0)])
    for bad in (np.nan, np.inf, -np.inf):
        for axis in (0, 1):
            r = ok.copy()
            r[2, axis] = bad
            feats = [([ok], 1), ([], 2), ([ok + 2, r], 3), ([ok], 4)]
            with pytest.raises(B2Error, match="feature 2 has a non-finite vertex"):
                ops.rasterize_layout(feats, 8)
    for v in (256, -1):
        with pytest.raises(B2Error, match="0..255"):
            ops.rasterize_layout([([ok], 1), ([ok], v)], 8)
    # a feature a trillion rows below the raster: no scanlines, no integer overflow
    L = ops.rasterize_layout([([ok], 1), (_zero_row_feature("far below", 8, 8), 2), ([ok], 3)], 8)
    assert L.job_off.tolist()[1:] == [5, 5, 10] and L.miny.dtype == np.int32


# ------------------------------------------------------------------------------------------------ GPU
def _gpu(feats, size, bg, at, dev):
    from dl_image_segmentation_b200 import ops
    return ops.rasterize_polygons(feats, size, bg, at, device=dev).cpu().numpy()


def _same_as_oracle(layers, dev, bg=255):
    for name, feats, size in layers:
        for at in (True, False):
            got, want = _gpu(feats, size, bg, at, dev), orr.rasterize(feats, size, bg, at)
            assert got.shape == want.shape and np.array_equal(got, want), (name, at, np.argwhere(got != want)[:5].tolist())


@pytest.mark.gpu
def test_gpu_centre_fill_equals_exact_reference(dev):
    for name, feats, (H, W) in _lattice_layers():
        got = _gpu(feats, (H, W), 255, False, dev)
        want = _exact_fill(feats, H, W, 255)
        assert np.array_equal(got, want), (name, np.argwhere(got != want)[:5].tolist())
        got, want = _gpu(feats, (H, W), 255, True, dev), orr.rasterize(feats, (H, W), 255, True)
        assert np.array_equal(got, want), (name, "all_touched", np.argwhere(got != want)[:5].tolist())


@pytest.mark.gpu
def test_gpu_gdal_shortcuts_and_ulp_edges(dev):
    _same_as_oracle(_shortcut_layers(), dev)


@pytest.mark.gpu
def test_gpu_clipping_and_far_vertices(dev):
    _same_as_oracle(_clip_layers(), dev, bg=0)


@pytest.mark.gpu
def test_gpu_raster_shapes(dev):
    _same_as_oracle(_shape_layers(), dev)
    rng = np.random.default_rng(4096)
    feats = [([_star(rng, rng.uniform(500, 3600, 2), 1800.0, 1500.0, 9)], 10 + f) for f in range(3)]
    feats.append(([np.array([(-100.0, 2047.5), (4200.0, 2047.5), (2048.0, 4200.0), (-100.0, 2047.5)])], 99))
    _same_as_oracle([("4096x4096", feats, (4096, 4096))], dev)


@pytest.mark.gpu
def test_gpu_burn_order(dev):
    _same_as_oracle([("5000 overlapping", _overlap_layer(), (96, 96))], dev, bg=17)
    _same_as_oracle(_order_layers(), dev, bg=200)


@pytest.mark.gpu
def test_gpu_dropin_on_the_tiles_own_grid(dev, tmp_path):
    """create_label_array_for_tile on GeoJSON layers whose map coordinates are whole and half pixels of the tile, and on
    features whose map coordinates are one ulp either side of such points (decimal round trips through other tools): the
    inverse geotransform then lands pixel coordinates next to integers and half-integers, not on them."""
    import dl_image_segmentation_b200 as pkg
    rng = np.random.default_rng(60)
    for i, (px, gt0, gt3, epsg) in enumerate(((0.5, 499680.0, 5300360.0, 32643), (10.0, 499680.0, 5300360.0, 32643),
                                              (30.0, 304980.0, 4430010.0, 32617), (60.0, 600000.0, 5000040.0, 32633),
                                              (10.0, 699960.0, 7500000.0, 32723), (30.0, 210000.0, 8999970.0, 32755))):
        class Tile:
            tilesize, pad = 56, 4
        Tile.geotrans, Tile.epsg = (gt0, px, 0.0, gt3, 0.0, -px), epsg
        gt = Tile.geotrans
        feats = []
        for f in range(24):
            start = rng.integers(-16, 144, 2) / 4.0
            rings = [_lattice_ring(rng, int(rng.integers(3, 9)), start, dmax=8.0) * 2.0]
            rings = [np.vstack([r, r[:1]]) for r in rings]
            feats.append((rings, int(rng.integers(0, 256))))
        for name, rings in _hand_shapes()[:10]:
            feats.append(([r * 2.0 + rng.integers(-4, 40) for r in rings], int(rng.integers(0, 256))))
        to_map = lambda r: np.stack([gt[0] + r[:, 0] * gt[1], gt[3] + r[:, 1] * gt[5]], 1)
        ulp = lambda m: np.nextafter(m, np.where(rng.random(m.shape) < 0.5, -np.inf, np.inf))
        gj = {"type": "FeatureCollection", "features": [
            {"type": "Feature", "properties": {"cls": v},
             "geometry": {"type": "Polygon", "coordinates": [(ulp(to_map(r)) if f % 3 == 2 else to_map(r)).tolist()
                                                             for r in rings]}} for f, (rings, v) in enumerate(feats)]}
        path = tmp_path / ("grid%d.geojson" % i)
        path.write_text(json.dumps(gj))
        layer = pkg.read_geojson_layer(str(path))
        pxs = np.concatenate([orr.to_pixel_space(r, gt) for rings, _ in layer for r in rings])
        assert (pxs * 2 == np.round(pxs * 2)).mean() > 0.5 and (np.abs(pxs * 2 - np.round(pxs * 2)) < 1e-6).all()
        assert (pxs * 2 != np.round(pxs * 2)).sum() > 20
        for attrib in ("cls", None):
            got = pkg.create_label_array_for_tile(Tile, str(path), attrib_to_burn=attrib, background_value=255, device=dev)
            want = orr.create_label_array_for_tile(56, 4, gt, layer, attrib, 255)
            assert np.array_equal(got.cpu().numpy(), want), (px, epsg, attrib, int((got.cpu().numpy() != want).sum()))


@pytest.mark.gpu
def test_gpu_layer_scale_workspace(dev):
    """2 000 small features and a 4 096-vertex one on a 512 x 512 tile, beside a 200 000-vertex feature off the tile's rows:
    burnt like the oracle, with less than 64 MiB of device memory beyond the owner and output buffers."""
    import torch
    from dl_image_segmentation_b200 import ops
    feats = _layer_scale()
    ops.rasterize_polygons(feats[:3], 512, 255, device=dev)             # context and module loaded outside the window
    torch.cuda.synchronize(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    got = ops.rasterize_polygons(feats, 512, 255, device=dev)
    torch.cuda.synchronize(dev)
    extra = torch.cuda.max_memory_allocated(dev) - base - 5 * 512 * 512
    assert extra < (64 << 20), extra
    want = orr.rasterize(feats, 512, 255, True)
    assert np.array_equal(got.cpu().numpy(), want)
    assert (want == 43).sum() > 50_000 and (want != 255).sum() > (want == 43).sum()


@pytest.mark.gpu
def test_gpu_far_feature_and_bad_input(dev):
    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    rng = np.random.default_rng(12)
    feats = _stars(rng, 10, 48, 48)
    far = (_zero_row_feature("far below", 48, 48), 77)
    for at in (True, False):
        want = orr.rasterize(feats, 48, 255, at)
        for k in (0, 5, 10):
            assert np.array_equal(_gpu(feats[:k] + [far] + feats[k:], 48, 255, at, dev), want), (at, k)
    ok = np.array([(1.0, 1.0), (6.0, 1.5), (3.0, 5.0), (1.0, 1.0)])
    for bad in (np.nan, np.inf, -np.inf):
        for axis in (0, 1):
            r = ok.copy()
            r[1, axis] = bad
            for at in (True, False):
                with pytest.raises(B2Error, match="feature 2 has a non-finite vertex"):
                    ops.rasterize_polygons([([ok], 1), ([ok], 2), ([r], 3)], 8, 0, at, device=dev)
    for v in (256, -1):
        with pytest.raises(B2Error):
            ops.rasterize_polygons([([ok], 1), ([ok], v)], 8, 0, device=dev)


@pytest.mark.gpu
def test_gpu_dropin_non_finite_vertices(dev):
    """In the tile's CRS a non-finite vertex is an error; in lon/lat a vertex that cannot be projected drops its feature
    with a warning, as OGR refuses to transform it."""
    import dl_image_segmentation_b200 as pkg
    from dl_image_segmentation_b200._lib import B2Error

    class Tile:
        tilesize, pad, epsg = 28, 2, 32643
        geotrans = (499680.0, 10.0, 0.0, 5300360.0, 0.0, -10.0)
    sq = np.array([(499700.0, 5300340.0), (499900.0, 5300340.0), (499900.0, 5300140.0), (499700.0, 5300340.0)])
    bad = sq.copy()
    bad[1, 0] = np.nan
    with pytest.raises(B2Error, match="feature 1 has a non-finite vertex"):
        pkg.create_label_array_for_tile(Tile, [([sq], {}), ([bad], {})], device=dev)
    lonlat = np.array([(75.0, 47.85), (75.002, 47.85), (75.001, 47.851), (75.0, 47.85)])
    nan = lonlat.copy()
    nan[2, 1] = np.nan
    with pytest.warns(UserWarning, match="1 label feature"):
        got = pkg.create_label_array_for_tile(Tile, [([lonlat], {}), ([nan], {})], device=dev, label_crs=4326)
    want = pkg.create_label_array_for_tile(Tile, [([lonlat], {})], device=dev, label_crs=4326)
    assert np.array_equal(got.cpu().numpy(), want.cpu().numpy())


@pytest.mark.gpu
def test_gpu_c_abi_refuses_rasters_of_2_31_pixels(dev):
    """The size check is on the host, before anything is launched: the buffers handed in here are far too small."""
    import torch
    from dl_image_segmentation_b200._lib import get_ctx, lib, ptr
    ctx = get_ctx(dev)
    owner = torch.empty(16, dtype=torch.int32, device=dev)
    out = torch.empty(16, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    l0 = ctx.launches
    for W, H in ((46341, 46341), (65536, 32768), (1 << 30, 2), (2, 1 << 30), (2 ** 31 - 1, 2), (0, 5), (5, -1)):
        rc = lib().b2_rasterize_polygons(ctx.handle, None, None, None, None, 0, None, None, 0, None, 0, W, H, 0, None,
                                         ptr(owner), None, ptr(out), ctx.stream())
        assert rc != 0 and b"bad raster size" in lib().b2_last_error(), (W, H)
    assert ctx.launches == l0
    torch.cuda.synchronize(dev)
