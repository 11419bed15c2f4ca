#!/usr/bin/env python3
"""Regenerate tests/golden/projection.npz.  Run from the repo root:  python tests/golden/gen_golden_projection.py

Reference values of the WGS84 transverse Mercator (EPSG:326zz / 327zz, UTM) for `ops.project_points` and the label
reprojection of `create_label_array_for_tile` — what PROJ's `utm` does for `gdal.RasterizeLayer` (reference
_descartes_img_chips.py:667-688).  PROJ is not installable here, and a reference that evaluated the same Krueger series as the
kernel would share its mistakes, so this module computes the projection from its definition, without any series:

  the transverse Mercator is the analytic continuation of the meridian arc, written as a function of the conformal latitude:
      y + i x = k0 * g(xi' + i eta'),   g(0) = 0,   g'(chi) = a cos(phi) / (sqrt(1 - e^2 sin^2 phi) cos(chi)),
  where phi(chi) inverts the conformal-latitude map (a complex root, found from chi) and (xi', eta') are the
  Gauss-Schreiber coordinates of the point.  g is a quadrature along the segment from 0 to xi' + i eta' at 30 digits;
  the inverse projection is a root of the forward map.

The forward and inverse points cover zones 1, 2, 30, 43, 59 and 60 in both hemispheres, latitudes -84..84 and +-89.99
(at a pole itself the integrand is 0/0), up to 10 degrees either side of the central meridian, the antimeridian (zone 1 at
179.5 E, zone 60 at 179.5 W) and the projection origin.  Two seeded label layers in longitude / latitude over 512 x 512 px
tiles at 10 m (448 px + 2 x 32 pad) come with their exact coordinates in the tiles' zones (43N; 23S) and, for the
northern one, in the neighbouring zone 44N.  About 0.4 s a point: the script spreads the points over the host's cores.
"""
import os
import sys
from multiprocessing import Pool

import mpmath as mp
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "projection.npz")

mp.mp.dps = 30
A = mp.mpf(6378137)
F = 1 / mp.mpf("298.257223563")
E2 = F * (2 - F)
E = mp.sqrt(E2)
K0 = mp.mpf("0.9996")
FE, FN_SOUTH = mp.mpf(500000), mp.mpf(10000000)

TILES = {  # name: (epsg, geotransform of a 448 + 2 x 32 px tile at 10 m)
    "n43": (32643, (499680.0, 10.0, 0.0, 5300360.0, 0.0, -10.0)),
    "s23": (32723, (291680.0, 10.0, 0.0, 7461120.0, 0.0, -10.0)),
}
TILE_PX = 512


def zone_of(epsg):
    """EPSG code -> (zone, south) of a WGS84 UTM zone."""
    zone, south = epsg % 100, epsg // 100 == 327
    assert epsg // 100 in (326, 327) and 1 <= zone <= 60, epsg
    return zone, south


def central_meridian(zone):
    return -183 + 6 * zone


def _psi(phi):
    """Isometric latitude (complex-capable)."""
    s = mp.sin(phi)
    return mp.atanh(s) - E * mp.atanh(E * s)


def _phi_of_chi(chi):
    """Geodetic latitude of conformal latitude chi: psi(phi) = atanh(sin chi), Newton from phi = chi."""
    target = mp.atanh(mp.sin(chi))
    dpsi = lambda p: (1 - E2) / ((1 - E2 * mp.sin(p) ** 2) * mp.cos(p))
    return mp.findroot(lambda p: _psi(p) - target, chi, solver="newton", df=dpsi)


def _dg(chi):
    phi = _phi_of_chi(chi)
    return A * mp.cos(phi) / (mp.sqrt(1 - E2 * mp.sin(phi) ** 2) * mp.cos(chi))


def _g(z):
    """The meridian arc as an analytic function of the (complex) conformal latitude."""
    if z == 0:
        return mp.mpc(0)
    return z * mp.quad(lambda t: _dg(t * z), [0, 1])


def _reduce_deg(d):
    """Degrees -> [-180, 180)."""
    d = mp.fmod(d, 360)
    return d - 360 if d >= 180 else (d + 360 if d < -180 else d)


def forward(lon, lat, epsg):
    """(lon, lat) degrees, WGS84 -> (easting, northing) m in UTM zone `epsg`, as mpf."""
    zone, south = zone_of(epsg)
    phi = mp.radians(mp.mpf(lat))
    dlam = mp.radians(_reduce_deg(mp.mpf(lon) - central_meridian(zone)))
    taup = mp.sinh(_psi(phi))                                # tan of the conformal latitude
    xip = mp.atan2(taup, mp.cos(dlam))                       # Gauss-Schreiber
    etap = mp.asinh(mp.sin(dlam) / mp.sqrt(taup ** 2 + mp.cos(dlam) ** 2))
    w = K0 * _g(mp.mpc(xip, etap))
    return FE + w.imag, w.real + (FN_SOUTH if south else 0)


def inverse(easting, northing, epsg):
    """(easting, northing) m in UTM zone `epsg` -> (lon in [-180, 180), lat) degrees, as mpf."""
    zone, south = zone_of(epsg)
    w = mp.mpc(mp.mpf(northing) - (FN_SOUTH if south else 0), mp.mpf(easting) - FE) / K0
    n = F / (2 - F)
    z0 = w * (1 + n) / (A * (1 + n ** 2 / 4))               # the rectifying radius, to start
    z = mp.findroot(lambda z: _g(z) - w, z0, solver="newton", df=_dg)
    xip, etap = z.real, z.imag
    taup = mp.sin(xip) / mp.sqrt(mp.sinh(etap) ** 2 + mp.cos(xip) ** 2)
    dlam = mp.atan2(mp.sinh(etap), mp.cos(xip))
    psi = mp.asinh(taup)
    phi = mp.findroot(lambda p: _psi(p) - psi, mp.atan(taup))
    return _reduce_deg(central_meridian(zone) + mp.degrees(dlam)), mp.degrees(phi)


def _fwd_job(a):
    lon, lat, epsg = a
    return tuple(float(v) for v in forward(lon, lat, epsg))


def _inv_job(a):
    e, n, epsg = a
    return tuple(float(v) for v in inverse(e, n, epsg))


# ---------------------------------------------------------------------------------------------------------- inputs
def forward_inputs(rng):
    pts = []
    for zone in (1, 2, 30, 43, 59, 60):
        lam0 = central_meridian(zone)
        for south in (False, True):
            epsg = (32700 if south else 32600) + zone
            for _ in range(22):
                lat = rng.uniform(0.0, 84.0) * (-1 if south else 1)
                pts.append((lam0 + rng.uniform(-10.0, 10.0), lat, epsg))
            pts.append((lam0 + rng.uniform(-3.0, 3.0), -89.99 if south else 89.99, epsg))
            pts.append((lam0, 0.0, epsg))                                                  # the origin
            pts.append((lam0 + rng.uniform(-3.0, 3.0), rng.uniform(-5.0, 5.0), epsg))      # the other hemisphere's edge
    for south in (False, True):                                                            # across the antimeridian
        s = -1 if south else 1
        pts.append((179.5, s * 12.25, (32700 if south else 32600) + 1))
        pts.append((-179.5, s * 47.5, (32700 if south else 32600) + 60))
        pts.append((-180.0, s * 3.0, (32700 if south else 32600) + 1))
    lon = [p[0] for p in pts]
    wrap = [((lo + 180.0) % 360.0) - 180.0 for lo in lon]                                  # zone 1 / 60 wrap into range
    return [(w, p[1], p[2]) for w, p in zip(wrap, pts)]


def pair_inputs(rng, k=30):
    """Points near the 43 / 44 zone boundary (78 E), projected into both zones: the UTM -> UTM reference."""
    return [(rng.uniform(74.0, 82.0), rng.uniform(-60.0, 70.0)) for _ in range(k)]


def inverse_inputs(rng):
    pts = []
    for zone in (1, 2, 30, 43, 59, 60):
        for south in (False, True):
            epsg = (32700 if south else 32600) + zone
            for _ in range(7):
                n = rng.uniform(0.0, 9330000.0)
                pts.append((round(rng.uniform(166000.0, 834000.0), 3), round(1e7 - n if south else n, 3), epsg))
            pts.append((500000.0, 10000000.0 if south else 0.0, epsg))                     # the origin
    pts += [(500000.0, 9329000.0, 32660), (833000.0, 12000.0, 32601), (167000.0, 9988000.0, 32760),
            (710000.0, 5300000.0, 32643)]
    return pts


def star(rng, centre, rmin, rmax, k):
    ang = np.sort(rng.random(k)) * 2 * np.pi
    rad = rng.uniform(rmin, rmax, k)
    ring = np.stack([centre[0] + rad * np.cos(ang), centre[1] + rad * np.sin(ang)], 1)
    return np.vstack([ring, ring[:1]])


def random_layer(rng, n, size):
    """Seeded polygons in pixel space (tests/test_rasterize.py's layer): some over the tile's edge, holes, multi-polygons.
    -> (vertices (V, 2), ring_off (R + 1), feat_off (n + 1) into the rings, values (n))."""
    rings, feat_off, values = [], [0], []
    for f in range(n):
        c = rng.uniform(-0.1 * size, 1.1 * size, 2)
        shell = star(rng, c, 0.03 * size, 0.35 * size, int(rng.integers(3, 12)))
        fr = [shell]
        if f % 3 == 0:
            fr.append((c + (shell - c) * 0.45)[::-1].copy())
        if f % 5 == 4:
            fr.append(star(rng, rng.uniform(0, size, 2), 0.02 * size, 0.1 * size, 5))
        rings += fr
        feat_off.append(len(rings))
        values.append(int(rng.integers(0, 256)))
    ring_off = np.cumsum([0] + [len(r) for r in rings])
    return np.vstack(rings), ring_off, np.asarray(feat_off), np.asarray(values, np.uint8)


def lonlat_layer(px, epsg, geotrans, pool):
    """A pixel-space layer laid over the tile in longitude / latitude: the tile's centre and its local scale come from the
    exact inverse; the polygons are then placed in degrees (any such layer is a valid test input — the reference values
    are the exact forward projections of these degrees)."""
    gt = geotrans
    cx, cy = gt[0] + gt[1] * TILE_PX / 2, gt[3] + gt[5] * TILE_PX / 2
    (lon_c, lat_c), (lon_e, _), (_, lat_n) = pool.map(_inv_job, [(cx, cy, epsg), (cx + 1000.0, cy, epsg),
                                                                 (cx, cy + 1000.0, epsg)])
    dlon, dlat = (lon_e - lon_c) / 1000.0, (lat_n - lat_c) / 1000.0      # degrees per metre (east, north)
    mx, my = (px[:, 0] - TILE_PX / 2) * gt[1], (px[:, 1] - TILE_PX / 2) * gt[5]
    return np.stack([lon_c + mx * dlon, lat_c + my * dlat], 1)


def main():
    rng = np.random.default_rng(20261022)
    out = {}
    with Pool(os.cpu_count()) as pool:
        fwd = forward_inputs(rng)
        pairs = pair_inputs(rng)
        fwd += [(lo, la, 32643) for lo, la in pairs] + [(lo, la, 32644) for lo, la in pairs]
        out["fwd_lonlat"] = np.array([p[:2] for p in fwd])
        out["fwd_epsg"] = np.array([p[2] for p in fwd], np.int32)
        out["fwd_utm"] = np.array(pool.map(_fwd_job, fwd))
        out["pair_idx"] = len(fwd) - 2 * len(pairs) + np.stack([np.arange(len(pairs)), len(pairs) + np.arange(len(pairs))], 1)
        print("forward", len(fwd), file=sys.stderr)
        inv = inverse_inputs(rng)
        out["inv_utm"] = np.array([p[:2] for p in inv])
        out["inv_epsg"] = np.array([p[2] for p in inv], np.int32)
        out["inv_lonlat"] = np.array(pool.map(_inv_job, inv))
        print("inverse", len(inv), file=sys.stderr)
        for name, (epsg, gt) in TILES.items():
            px, ring_off, feat_off, values = random_layer(rng, 24, TILE_PX)
            ll = lonlat_layer(px, epsg, gt, pool)
            out[name + "_geotrans"] = np.array(gt)
            out[name + "_lonlat"] = ll
            out[name + "_ring_off"], out[name + "_feat_off"], out[name + "_values"] = ring_off, feat_off, values
            zones = [epsg] + ([epsg + 1] if name == "n43" else [])
            for z in zones:
                out["%s_utm%d" % (name, z)] = np.array(pool.map(_fwd_job, [(lo, la, z) for lo, la in ll]))
            print(name, len(ll), "vertices", file=sys.stderr)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, file=sys.stderr)


if __name__ == "__main__":
    main()
