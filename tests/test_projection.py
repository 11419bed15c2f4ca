"""Label layers in another CRS than the tile's: `ops.project_points` (b2_project_points, WGS84 transverse Mercator / UTM)
and the reprojection `create_label_array_for_tile` does before it burns, as gdal.RasterizeLayer does
(`_descartes_img_chips.py:667-688`).

The reference values come from tests/golden/gen_golden_projection.py, which computes the projection from its definition (a
complex quadrature of the meridian arc over the conformal latitude, 30 digits) and shares no series with the kernel.
CPU: that reference is pinned on the central meridian against an independent meridian-arc quadrature and recomputed live on
a few committed points; the layer-CRS rules.  GPU: the kernel against the committed points; whole label chips bit-identical
with the rasteriser's oracle on the exactly projected coordinates.
"""
import datetime as dt
import importlib.util
import json
import os
import warnings

import mpmath as mp
import numpy as np
import pytest

from oracle import rasterize as orr

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G = np.load(os.path.join(GOLD, "projection.npz"))


def _gen():
    spec = importlib.util.spec_from_file_location("gen_golden_projection", os.path.join(GOLD, "gen_golden_projection.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _dc():
    from dl_image_segmentation_b200 import _descartes_img_chips as dc
    return dc


# ---------------------------------------------------------------------------------------------------------- CPU
def test_reference_projection_on_the_central_meridian_is_k0_times_the_meridian_arc():
    g = _gen()
    a, e2 = mp.mpf(6378137), g.E2
    for lat in (0.0, 12.5, -33.0, 45.0, 70.25, -84.0):
        phi = mp.radians(lat)
        arc = mp.quad(lambda p: a * (1 - e2) / (1 - e2 * mp.sin(p) ** 2) ** 1.5, [0, phi])
        for epsg in (32643, 32743):
            e, n = g.forward(75.0, lat, epsg)
            assert abs(e - 500000) < 1e-9
            assert abs(n - (g.K0 * arc + (10000000 if epsg == 32743 else 0))) < 1e-9, (lat, epsg)


def test_committed_projection_points_are_what_the_reference_computes():
    g = _gen()
    for i in (0, 23, 100, 200, len(G["fwd_epsg"]) - 1):
        lon, lat = G["fwd_lonlat"][i]
        got = np.array([float(v) for v in g.forward(lon, lat, int(G["fwd_epsg"][i]))])
        assert np.abs(got - G["fwd_utm"][i]).max() < 1e-9, i
    for i in (3, 50):
        e, n = G["inv_utm"][i]
        got = np.array([float(v) for v in g.inverse(e, n, int(G["inv_epsg"][i]))])
        assert np.abs(got - G["inv_lonlat"][i]).max() < 1e-12, i
    origin = G["fwd_lonlat"][:, 1] == 0.0                          # (central meridian, equator) -> (500 000, 0)
    assert origin.sum() >= 12 and np.array_equal(G["fwd_utm"][origin] % 10000000, [[500000.0, 0.0]] * int(origin.sum()))


def test_geojson_crs_member_spellings():
    dc = _dc()
    name = lambda s: {"crs": {"type": "name", "properties": {"name": s}}}
    assert dc.geojson_crs_epsg({}) is None
    assert dc.geojson_crs_epsg(name("EPSG:4326")) == 4326
    assert dc.geojson_crs_epsg(name("urn:ogc:def:crs:EPSG::32643")) == 32643
    assert dc.geojson_crs_epsg(name("urn:ogc:def:crs:OGC:1.3:CRS84")) == 4326
    assert dc.geojson_crs_epsg(name("epsg:32723")) == 32723
    for bad in ("EPSG:", "urn:ogc:def:crs:EPSG::x", "WGS 84"):
        with pytest.raises(dc.B2Error, match="not supported"):
            dc.geojson_crs_epsg(name(bad))
    with pytest.raises(dc.B2Error, match="named CRSs"):
        dc.geojson_crs_epsg({"crs": {"type": "link", "properties": {"href": "x"}}})


def test_label_layer_crs_resolution():
    dc = _dc()
    lonlat = [([np.array([[75.1, 47.8], [75.2, 47.8], [75.2, 47.9], [75.1, 47.8]])], {})]
    utm = [([np.array([[499680.0, 5300360.0], [504800.0, 5300360.0], [504800.0, 5295240.0], [499680.0, 5300360.0]])], {})]
    # label_crs first, then the crs member, then the no-crs rule
    assert dc.label_layer_epsg(32643, 4326, 32644, utm) == 4326
    assert dc.label_layer_epsg(32643, "EPSG:32644", None, lonlat) == 32644
    assert dc.label_layer_epsg(32643, None, 32644, lonlat) == 32644
    assert dc.label_layer_epsg(32643, None, None, lonlat) == 4326
    assert dc.label_layer_epsg(32743, None, None, lonlat) == 4326
    assert dc.label_layer_epsg(32643, None, None, utm) == 32643            # a layer in the tile's CRS, as before
    assert dc.label_layer_epsg(0, None, None, lonlat) == 0                   # tile CRS unknown: coordinates as they are
    assert dc.label_layer_epsg(32643, None, None, []) == 32643
    # declared CRSs outside 4326 / WGS84 UTM, and labels that would need projecting onto a tile that is not UTM
    for crs in (3857, "EPSG:32661", "EPSG:32600", 27700):
        with pytest.raises(dc.B2Error, match="EPSG:%d" % (crs if isinstance(crs, int) else int(crs[5:]))):
            dc.label_layer_epsg(32643, crs, None, lonlat)
    with pytest.raises(dc.B2Error, match="EPSG:3857"):
        dc.label_layer_epsg(32643, None, 3857, lonlat)
    with pytest.raises(dc.B2Error, match="unknown CRS"):
        dc.label_layer_epsg(0, None, 4326, lonlat)
    with pytest.raises(dc.B2Error, match="EPSG:3857"):
        dc.label_layer_epsg(3857, 32643, None, utm)


# ---------------------------------------------------------------------------------------------------------- GPU
def _ops():
    from dl_image_segmentation_b200 import ops
    return ops


@pytest.mark.gpu
def test_gpu_forward_matches_the_reference(dev):
    ops = _ops()
    for epsg in np.unique(G["fwd_epsg"]):
        m = G["fwd_epsg"] == epsg
        got = ops.project_points(G["fwd_lonlat"][m], 4326, int(epsg), device=dev)
        assert got.is_cuda and got.dtype.is_floating_point and tuple(got.shape) == (int(m.sum()), 2)
        d = np.abs(got.cpu().numpy() - G["fwd_utm"][m]).max()
        assert d <= 1e-6, (int(epsg), d)


@pytest.mark.gpu
def test_gpu_inverse_matches_the_reference(dev):
    ops = _ops()
    for epsg in np.unique(G["inv_epsg"]):
        m = G["inv_epsg"] == epsg
        got = ops.project_points(G["inv_utm"][m], int(epsg), 4326, device=dev).cpu().numpy()
        assert np.abs(got - G["inv_lonlat"][m]).max() <= 1e-11, int(epsg)
        assert (got[:, 0] >= -180.0).all() and (got[:, 0] < 180.0).all()


@pytest.mark.gpu
def test_gpu_zone_to_zone_and_round_trip(dev):
    import torch
    ops = _ops()
    a, b = G["pair_idx"][:, 0], G["pair_idx"][:, 1]
    u43 = torch.from_numpy(G["fwd_utm"][a])                           # a CPU tensor is taken too
    assert np.abs(ops.project_points(u43, 32643, 32644, device=dev).cpu().numpy() - G["fwd_utm"][b]).max() <= 1e-6
    assert np.abs(ops.project_points(G["fwd_utm"][b], 32644, 32643, device=dev).cpu().numpy() - G["fwd_utm"][a]).max() <= 1e-6
    south = G["fwd_utm"][a] + [0.0, 10000000.0]                        # the same points in 43S: only the false northing moves
    assert np.abs(ops.project_points(u43, 32643, 32743, device=dev).cpu().numpy() - south).max() <= 1e-6
    for epsg in np.unique(G["fwd_epsg"]):
        m = G["fwd_epsg"] == epsg
        ll = ops.project_points(G["fwd_utm"][m], int(epsg), 4326, device=dev)
        back = ops.project_points(ll, 4326, int(epsg), device=dev).cpu().numpy()
        assert np.abs(back - G["fwd_utm"][m]).max() <= 1e-6, int(epsg)
    same = ops.project_points(G["fwd_utm"][a], 32643, 32643, device=dev).cpu().numpy()
    assert np.array_equal(same, G["fwd_utm"][a])                      # equal codes copy
    assert tuple(ops.project_points(np.zeros((0, 2)), 4326, 32643, device=dev).shape) == (0, 2)


@pytest.mark.gpu
def test_gpu_invalid_vertices_and_codes(dev):
    ops = _ops()
    nan, inf = float("nan"), float("inf")
    bad = np.array([[nan, 10.0], [75.0, inf], [75.0, 90.5], [75.0, -91.0], [165.0, 10.0], [-15.0, 0.0], [-105.0, 45.0]])
    out = ops.project_points(bad, 4326, 32643, device=dev).cpu().numpy()
    assert np.isnan(out).all()
    ok = np.array([[75.0, 90.0], [75.0, -90.0], [164.9, 0.0]])        # the poles, and just under 90 degrees east
    assert np.isfinite(ops.project_points(ok, 4326, 32643, device=dev).cpu().numpy()).all()
    far = ops.project_points(np.array([[500000.0, 5000000.0], [nan, 0.0]]), 32601, 32631, device=dev).cpu().numpy()
    assert np.isnan(far).all()                                         # 180 degrees apart; not finite
    assert np.isnan(ops.project_points(np.array([[inf, 0.0]]), 32643, 4326, device=dev).cpu().numpy()).all()
    for src, dst in ((4326, 3857), (3857, 32643), (32600, 4326), (32661, 4326), (4326, 32761), (32543, 4326)):
        with pytest.raises(ops.B2Error, match="EPSG:%d" % (dst if src == 4326 else src)):
            ops.project_points(ok, src, dst, device=dev)
    with pytest.raises(ops.B2Error, match="float64"):
        ops.project_points(ok.astype(np.float32), 4326, 32643, device=dev)


def _layer(name, xy):
    ro, fo, v = G[name + "_ring_off"], G[name + "_feat_off"], G[name + "_values"]
    rings = [xy[ro[i]:ro[i + 1]] for i in range(len(ro) - 1)]
    return [(rings[fo[f]:fo[f + 1]], {"cls": int(v[f])}) for f in range(len(fo) - 1)]


def _geojson(layer, crs=None):
    gj = {"type": "FeatureCollection", "features": [
        {"type": "Feature", "properties": props,
         "geometry": {"type": "Polygon", "coordinates": [r.tolist() for r in rings]} if len(rings) == 1 else
                     {"type": "MultiPolygon", "coordinates": [[r.tolist()] for r in rings]}} for rings, props in layer]}
    if crs is not None:
        gj["crs"] = {"type": "name", "properties": {"name": crs}}
    return gj


def _tile(name):
    epsg = {"n43": 32643, "s23": 32723}[name]

    class Tile:
        key = "448:32:10.0:%d:%s" % (epsg % 100, name)
        tilesize, pad, geotrans = 448, 32, tuple(G[name + "_geotrans"])
    Tile.epsg = epsg
    return Tile


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n43", "s23"])
def test_gpu_lonlat_labels_are_burnt_where_the_exact_projection_puts_them(dev, tmp_path, name):
    """cfg3 tile geometry (448 px + 2 x 32 pad, 10 m) in zone 43N and 23S; a seeded lon/lat layer (holes, multi-polygons,
    polygons over the tile's edge).  The kernel's coordinates are within nanometres of the reference's, ~1e-10 px: the
    seed of the committed layers puts no crossing that close to a pixel boundary, so the chips are bit-identical."""
    import dl_image_segmentation_b200 as pkg
    tile = _tile(name)
    utm = _layer(name, G["%s_utm%d" % (name, tile.epsg)])
    want = orr.create_label_array_for_tile(448, 32, tile.geotrans, utm, "cls", 255)
    assert (want != 255).mean() > 0.3 and len(np.unique(want)) > 10
    lonlat = _layer(name, G[name + "_lonlat"])
    layers = {"no crs": _geojson(lonlat), "CRS84": _geojson(lonlat, "urn:ogc:def:crs:OGC:1.3:CRS84"),
              "EPSG::4326": _geojson(lonlat, "urn:ogc:def:crs:EPSG::4326"), "own UTM": _geojson(utm)}
    if name == "n43":
        layers["zone 44"] = _geojson(_layer(name, G["n43_utm32644"]), "EPSG:32644")
    for what, gj in layers.items():
        path = tmp_path / ("%s.geojson" % what.replace(" ", "_").replace(":", "_"))
        path.write_text(json.dumps(gj))
        got = pkg.create_label_array_for_tile(tile, str(path), attrib_to_burn="cls", background_value=255, device=dev)
        assert got.is_cuda and np.array_equal(got.cpu().numpy(), want), (name, what, int((got.cpu().numpy() != want).sum()))
    got = pkg.create_label_array_for_tile(tile, lonlat, attrib_to_burn="cls", device=dev, label_crs=4326)
    assert np.array_equal(got.cpu().numpy(), want)
    got = pkg.create_label_array_for_tile(tile, [[], lonlat], attrib_to_burn="cls", layer_idx=1, device=dev, label_crs="EPSG:4326")
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.gpu
def test_gpu_unprojectable_feature_is_skipped_with_a_warning(dev):
    import dl_image_segmentation_b200 as pkg
    tile = _tile("n43")
    lonlat = _layer("n43", G["n43_lonlat"])
    far = ([np.array([[170.0, 10.0], [171.0, 10.0], [171.0, 11.0], [170.0, 10.0]])], {"cls": 7})   # 95 degrees off zone 43
    with pytest.warns(UserWarning, match="1 label feature"):
        got = pkg.create_label_array_for_tile(tile, lonlat[:5] + [far] + lonlat[5:], attrib_to_burn="cls", device=dev, label_crs=4326)
    want = orr.create_label_array_for_tile(448, 32, tile.geotrans, _layer("n43", G["n43_utm32643"]), "cls", 255)
    assert np.array_equal(got.cpu().numpy(), want)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        pkg.create_label_array_for_tile(tile, lonlat, attrib_to_burn="cls", device=dev, label_crs=4326)
    with pytest.raises(pkg._descartes_img_chips.B2Error, match="unknown CRS"):
        class NoCrs:
            tilesize, pad, geotrans = 448, 32, tile.geotrans
        pkg.create_label_array_for_tile(NoCrs, lonlat, device=dev, label_crs=4326)


@pytest.mark.gpu
def test_gpu_create_chips_for_tile_with_a_lonlat_label_file(dev, tmp_path):
    import dl_image_segmentation_b200 as pkg
    from dl_image_segmentation_b200 import _descartes_img_chips as dc
    from oracle import imagecodecs as oic
    tile = _tile("n43")
    path = tmp_path / "labels.geojson"
    path.write_text(json.dumps(_geojson(_layer("n43", G["n43_lonlat"]))))
    rng = np.random.default_rng(3)
    src = dc.SyntheticSceneSource()
    stack = rng.integers(0, 4000, (2, 512, 512, 3)).astype(np.uint16)
    src.add(tile, "landsat:LC08:PRE:TOAR", dc.SceneStack(stack, np.ones((2, 512, 512), np.uint8),
                                                         [dt.date(2020, 1, 1), dt.date(2020, 2, 1)], [0.1, 0.2]))
    job = pkg.DLTileJobConfig(tile, str(tmp_path / "out"), "landsat:LC08:PRE:TOAR", dt.date(2020, 2, 1), str(path), label_attr="cls")
    ret, img_file, lbl_file = pkg.create_chips_for_tile(job, scene_source=src, device=dev)
    assert ret is job and img_file is not None
    got = oic.decode_image(open(lbl_file, "rb").read(), png_as_tf=False)
    want = orr.create_label_array_for_tile(448, 32, tile.geotrans, _layer("n43", G["n43_utm32643"]), "cls", 255)
    assert np.array_equal(got.reshape(want.shape), want) and (want != 255).any()
