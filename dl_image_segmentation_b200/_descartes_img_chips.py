"""Per-tile compositors — B200 drop-in for the array half of the reference's ``_descartes_img_chips.py``.

The reference fetches its time stacks from the Descartes Labs cloud service (``dl.scenes.search``,
``SceneCollection.stack/mosaic`` — network, out of scope) and then does the per-pixel arithmetic with
NumPy (``:562-567``) or leaves it to the remote mosaic call (``:622-626``).  Here the stacks come from an
injectable *scene source* (synthetic stacks in tests/bench) and the arithmetic runs on the GPU:

  ``median_composite``       = ``:562-567``  -> ``b2_median_composite_u16``
  ``nearest_date_mosaic``    = ``:603-626`` + ``:461-469`` -> ``b2_nearest_date_mosaic``
  ``create_cloudmasked_s2_array`` / ``create_img_array_for_tile`` / ``stack_products_for_tile`` keep the
  reference signatures (``:521-522, :571-572, :472``) with one extra trailing kwarg ``scene_source``.

Behaviour kept: no scenes after the search filter -> ``None`` (``:554-555,614-615``); date filter is
``min_date <= date < max_date`` (``start_datetime``/``end_datetime`` ``:603-606``); cloud filter strict ``<``
(``:610``); ties in ``abs(date - reference_date)`` go to the later scene of the search order (stable
``sorted(reverse=True)`` ``:623``, last painted wins ``:619-621``); median result is float64 + mask.
"""
import datetime as _dt

import numpy as np
import torch

from . import ops
from ._lib import B2Error


_SIGNED_VIEW = {torch.uint16: torch.int16, torch.uint32: torch.int32, torch.uint64: torch.int64}
_NP_NAME = {torch.uint8: "uint8", torch.int8: "int8", torch.uint16: "uint16", torch.int16: "int16", torch.uint32: "uint32",
            torch.int32: "int32", torch.uint64: "uint64", torch.int64: "int64", torch.float16: "float16",
            torch.float32: "float32", torch.float64: "float64", torch.bool: "bool"}
_TORCH_OF = {v: k for k, v in _NP_NAME.items()}


def _moved(t, fn):
    """Apply a pure data-movement op (where / index_select / cat) to a tensor whose dtype torch may not implement it for
    (uint16 / uint32): run it on the same-width signed view and view the result back."""
    sv = _SIGNED_VIEW.get(t.dtype)
    return fn(t) if sv is None else fn(t.view(sv)).view(t.dtype)


def _cast(t, dtype):
    """.astype(dtype) with NumPy's value semantics for the integer widenings np.dstack can ask for."""
    if t.dtype == dtype:
        return t
    if t.dtype in _SIGNED_VIEW:                                   # unsigned source: widen through int64 (zero-extended)
        bits = t.element_size() * 8
        wide = t.view(_SIGNED_VIEW[t.dtype]).to(torch.int64)
        wide = torch.where(wide < 0, wide + (1 << bits), wide) if bits < 64 else wide
        t = wide
    if dtype in _SIGNED_VIEW:                                     # unsigned target: values fit, store through the signed twin
        return t.to(torch.int64).to(_SIGNED_VIEW[dtype]).view(dtype)
    return t.to(dtype)


class MaskedResult:
    """np.ma-compatible pair living on the device: ``data`` (H,W,B) and boolean ``mask`` (True = masked)."""

    def __init__(self, data, mask):
        self.data, self.mask = data, mask
        self.shape, self.dtype = tuple(data.shape), data.dtype

    def to_masked_array(self):
        return np.ma.MaskedArray(self.data.cpu().numpy(), mask=self.mask.cpu().numpy())

    def filled(self, fill_value=0):
        fill = torch.from_numpy(np.asarray(fill_value).astype(_NP_NAME[self.data.dtype]).reshape(1)).to(self.data.device)
        sv = _SIGNED_VIEW.get(self.data.dtype)
        if sv is not None:
            fill = fill.view(sv)
        return _moved(self.data, lambda d: torch.where(self.mask, fill.reshape(()), d))


class SceneStack:
    """What a scene source returns for one geocontext/product: the scenes in SEARCH ORDER."""

    def __init__(self, stack, valid, dates, cloud_fraction=None, nodata_mask=None):
        self.stack, self.valid = stack, valid              # (T,H,W,B), (T,H,W) uint8 (1 = usable pixel)
        self.dates = list(dates)                           # datetime.date / datetime.datetime per scene
        self.cloud_fraction = None if cloud_fraction is None else list(cloud_fraction)
        self.nodata_mask = nodata_mask                     # optional (T,H,W,B), non-zero = masked


class SyntheticSceneSource:
    """Dict-backed stand-in for ``dl.scenes.search``: ``{(ctx_key, product): SceneStack}``."""

    def __init__(self, table=None):
        self.table = dict(table or {})

    def add(self, ctx, product, scene_stack):
        self.table[(_ctx_key(ctx), product)] = scene_stack

    def search(self, ctx, product):
        return self.table.get((_ctx_key(ctx), product))


def _ctx_key(ctx):
    return getattr(ctx, "key", ctx if isinstance(ctx, (str, int, tuple)) else id(ctx))


def _to_day(d):
    if d is None:
        return None
    if isinstance(d, _dt.datetime):
        d = d.date()
    if isinstance(d, _dt.date):
        return d.toordinal()
    return int(d)


def _get_scene_date_diff_mapper(reference_date):
    """Returns a function giving |scene date - reference date| (reference :461-469)."""
    ref = _to_day(reference_date)

    def get_date_diff(scene_date):
        return abs(_to_day(scene_date) - ref)
    return get_date_diff


def _select_scenes(stack, valid, keep):
    """View (contiguous run) or gather of the scenes that survive a search filter — data movement only."""
    keep = list(keep)
    if keep == list(range(keep[0], keep[-1] + 1)):
        return stack[keep[0]:keep[-1] + 1], valid[keep[0]:keep[-1] + 1]
    ix = torch.as_tensor(keep, dtype=torch.int64, device=stack.device)
    return _moved(stack, lambda t: t.index_select(0, ix)), _moved(valid, lambda t: t.index_select(0, ix))


def median_composite(stack, valid, nodata_mask=None, device=None):
    """Cloud-masked per-pixel median over axis 0 -> MaskedResult (float64).  Replaces reference :562-567."""
    out, mask = ops.median_composite(stack, valid, nodata_mask, device)
    return MaskedResult(out, mask)


def nearest_date_mosaic(stack, valid, scene_dates, scene_cloud_fraction, reference_date, min_date=None, max_date=None,
                        max_cloud_fraction=None, device=None, return_source_index=False):
    """Nearest-to-reference-date mosaic of ONE chip -> MaskedResult, or None when no scene survives the filter."""
    T = len(scene_dates)
    day = np.asarray([_to_day(d) for d in scene_dates], dtype=np.int32).reshape(1, T)
    cf = np.zeros((1, T), dtype=np.float32) if scene_cloud_fraction is None else \
        np.asarray(scene_cloud_fraction, dtype=np.float32).reshape(1, T)
    if scene_cloud_fraction is None and max_cloud_fraction is not None:
        raise B2Error("max_cloud_fraction given but the scenes carry no cloud_fraction")
    out, mask, src, nel = ops.nearest_date_mosaic([stack], [valid], day, cf, _to_day(reference_date), _to_day(min_date),
                                                  _to_day(max_date), max_cloud_fraction, device=device)
    if int(nel.cpu()[0]) == 0:
        return None                                             # reference :614-615
    B = out.shape[-1]
    res = MaskedResult(out[0], mask[0].unsqueeze(-1).expand(-1, -1, B))
    return (res, src[0]) if return_source_index else res


def create_cloudmasked_s2_array(ctx, min_date=None, max_date=None, bands="red green blue", scene_source=None):
    """Cloud-free Sentinel-2 median mosaic for a geocontext (reference :521-568)."""
    if scene_source is None:
        raise B2Error("the Descartes Labs catalog is out of scope: pass scene_source=SyntheticSceneSource(...)")
    sc = scene_source.search(ctx, "sentinel-2:L1C")
    if sc is None or len(sc.dates) == 0:
        return None
    lo, hi = _to_day(min_date), _to_day(max_date)
    keep = [i for i, d in enumerate(sc.dates)
            if (lo is None or _to_day(d) >= lo) and (hi is None or _to_day(d) < hi)]
    if not keep:
        return None                                             # reference :554-555
    ctxd = ops.get_ctx(None)
    stack = ops.to_device(sc.stack, ctxd.device)
    valid = ops.to_device(sc.valid, ctxd.device)
    if valid.dim() == 4:
        valid = valid[..., 0]
    nd = None if sc.nodata_mask is None else ops.to_device(sc.nodata_mask, ctxd.device)
    if len(keep) != len(sc.dates):
        if nd is not None:
            nd = _select_scenes(nd, valid, keep)[0]
        stack, valid = _select_scenes(stack, valid, keep)
    nb = len(bands.split(" ")) if isinstance(bands, str) else len(bands)
    if stack.shape[-1] != nb:
        raise B2Error("scene source returned %d bands for bands=%r" % (stack.shape[-1], bands))
    return median_composite(stack.contiguous(), valid.contiguous(), None if nd is None else nd.contiguous())


def create_img_array_for_tile(ctx, product, reference_date, min_date=None, max_date=None, bands="red green blue",
                              max_cloud_fraction=None, scene_source=None):
    """Nearest-date mosaic for a geocontext (reference :571-629).  Any failure -> None (bare except, :628-629)."""
    if scene_source is None:
        raise B2Error("the Descartes Labs catalog is out of scope: pass scene_source=SyntheticSceneSource(...)")
    sc = scene_source.search(ctx, product)
    if sc is None or len(sc.dates) == 0:
        return None
    try:
        return nearest_date_mosaic(sc.stack, sc.valid, sc.dates, sc.cloud_fraction, reference_date, min_date, max_date,
                                   max_cloud_fraction)
    except Exception:
        return None


def stack_products_for_tile(ctx, products, bands_per_product, resampler="near", scene_source=None):
    """Per-product overlay mosaic (no filters, last scene wins) then band-concatenate (reference :472-518, np.dstack :516)."""
    if scene_source is None:
        raise B2Error("the Descartes Labs catalog is out of scope: pass scene_source=SyntheticSceneSource(...)")
    arrays = []
    for product in products:
        sc = scene_source.search(ctx, product)
        if sc is None or len(sc.dates) == 0:
            # the reference does not test for this (:512-513): SceneCollection.mosaic of an empty collection raises
            raise ValueError("This SceneCollection is empty (product %r)" % (product,))
        # plain mosaic(): scenes painted in search order == every scene at the same "distance", later index wins
        same_day = [0] * len(sc.dates)
        res = nearest_date_mosaic(sc.stack, sc.valid, same_day, None, 0)
        arrays.append(res.data)                     # kernel already wrote 0 where no scene is valid
    if len({a.dtype for a in arrays}) > 1:          # np.dstack promotes mixed dtypes by NumPy's rules (u16 + i16 -> int32)
        dt = np.result_type(*[np.dtype(_NP_NAME[a.dtype]) for a in arrays])
        arrays = [_cast(a, _TORCH_OF[dt.name]) for a in arrays]
    return _cat_last(arrays)


def _cat_last(arrays):
    sv = _SIGNED_VIEW.get(arrays[0].dtype)
    if sv is None:
        return torch.cat(arrays, dim=-1)
    return torch.cat([a.view(sv) for a in arrays], dim=-1).view(arrays[0].dtype)


# ------------------------------------------------------------------------------------------------ label rasterisation
def _load_geojson(path_or_dict):
    import json
    if isinstance(path_or_dict, dict):
        return path_or_dict
    with open(path_or_dict, "r") as f:
        return json.load(f)


def read_geojson_layer(path_or_dict):
    """A label layer from GeoJSON (the format of the reference's label data, .MISSING_LARGE_BLOBS): list of
    (rings, properties) per Polygon / MultiPolygon feature, in file order — what iterating the OGR layer yields.
    Coordinates are returned as they are, in the layer's CRS (geojson_crs_epsg)."""
    gj = _load_geojson(path_or_dict)
    feats = gj["features"] if gj.get("type") == "FeatureCollection" else [gj]
    layer = []
    for ft in feats:
        geom = ft.get("geometry") or {}
        if geom.get("type") == "Polygon":
            rings = [np.asarray(r, dtype=np.float64)[:, :2] for r in geom["coordinates"]]
        elif geom.get("type") == "MultiPolygon":
            rings = [np.asarray(r, dtype=np.float64)[:, :2] for poly in geom["coordinates"] for r in poly]
        else:
            continue                                            # RasterizeLayer burns nothing for an empty geometry
        layer.append((rings, ft.get("properties") or {}))
    return layer


_CRS84 = "URN:OGC:DEF:CRS:OGC:1.3:CRS84"


def _epsg_of_name(name):
    """'EPSG:n', 'urn:ogc:def:crs:EPSG::n' or the CRS84 URN (longitude / latitude on WGS84, = 4326) -> n."""
    u = str(name).strip().upper()
    if u == _CRS84:
        return 4326
    for prefix in ("EPSG:", "URN:OGC:DEF:CRS:EPSG::"):
        if u.startswith(prefix) and u[len(prefix):].isdigit():
            return int(u[len(prefix):])
    raise B2Error("label CRS %r is not supported (EPSG:4326, CRS84 or a WGS84 UTM zone EPSG:326zz / 327zz)" % (name,))


def geojson_crs_epsg(gj):
    """EPSG code of a GeoJSON object's ``crs`` member ({"type": "name", "properties": {"name": ...}}), None without one."""
    crs = gj.get("crs")
    if crs is None:
        return None
    name = (crs.get("properties") or {}).get("name") if isinstance(crs, dict) else None
    if name is None:
        raise B2Error("label CRS %r is not supported: only named CRSs ({'type': 'name', ...}) are read" % (crs,))
    return _epsg_of_name(name)


def _is_utm(epsg):
    return epsg // 100 in (326, 327) and 1 <= epsg % 100 <= 60


def label_layer_epsg(tile_epsg, label_crs=None, crs_member=None, layer=()):
    """The CRS a label layer is in, as RasterizeLayer would learn it from the layer's SRS: ``label_crs`` (an EPSG int or
    'EPSG:n') if given, else the GeoJSON ``crs`` member's code (geojson_crs_epsg), else — no CRS declared — longitude /
    latitude (4326) when the tile is in UTM and every coordinate lies in [-180, 180] x [-90, 90] (GeoJSON's default CRS; a
    UTM easting is never below ~160 km, so a layer in the tile's own CRS never passes), else the tile's CRS.  Raises B2Error
    for a declared CRS other than 4326 / WGS84 UTM, or a layer that needs projecting onto a tile that is not in UTM."""
    if label_crs is not None:
        epsg = int(label_crs) if isinstance(label_crs, (int, np.integer)) else _epsg_of_name(label_crs)
    else:
        epsg = crs_member
    if epsg is None:
        xy = [np.asarray(r, dtype=np.float64).reshape(-1, 2) for rings, _ in layer for r in rings]
        xy = np.concatenate(xy) if xy else np.zeros((0, 2))
        lonlat = len(xy) > 0 and bool((np.abs(xy[:, 0]) <= 180.0).all() and (np.abs(xy[:, 1]) <= 90.0).all())
        return 4326 if _is_utm(tile_epsg) and lonlat else tile_epsg
    if epsg != 4326 and not _is_utm(epsg):
        raise B2Error("label CRS EPSG:%d is not supported (EPSG:4326 or a WGS84 UTM zone EPSG:326zz / 327zz)" % epsg)
    if epsg != tile_epsg and not _is_utm(tile_epsg):
        raise B2Error("labels in EPSG:%d cannot be projected onto a tile in %s: only WGS84 UTM tiles are supported"
                      % (epsg, "EPSG:%d" % tile_epsg if tile_epsg else "an unknown CRS"))
    return epsg


def _project_layer(layer, src_epsg, dst_epsg, device):
    """Every vertex of the layer in one upload, one b2_project_points launch and one download; vertices only, as
    OGRGeometry::transform does (edges are not densified).  A feature with a vertex the projection is not valid for is
    dropped with a warning: OGR refuses to transform such a geometry, so it burns nothing."""
    rings = [np.asarray(r, dtype=np.float64).reshape(-1, 2) for rs, _ in layer for r in rs]
    if not rings:
        return layer
    xy = ops.project_points(np.concatenate(rings), src_epsg, dst_epsg, device=device).cpu().numpy()
    ring_end = np.cumsum([len(r) for r in rings])
    feat_end = np.cumsum([len(rs) for rs, _ in layer])
    nan_upto = np.concatenate([[0], np.cumsum(np.isnan(xy).any(axis=1))])          # NaN vertices before vertex i
    vert_end = np.concatenate([[0], ring_end])[feat_end]                             # first vertex after feature f
    bad = np.diff(np.concatenate([[0], nan_upto[vert_end]])) > 0
    projected = [xy[i:j] for i, j in zip([0] + ring_end[:-1].tolist(), ring_end.tolist())]
    out, at = [], 0
    for (rs, props), end, b in zip(layer, feat_end, bad):
        if not b:
            out.append((projected[at:end], props))
        at = end
    skipped = int(bad.sum())
    if skipped:
        import warnings
        warnings.warn("create_label_array_for_tile: %d label feature(s) have vertices that cannot be projected from EPSG:%d "
                      "to EPSG:%d; they are not burnt" % (skipped, src_epsg, dst_epsg))
    return out


def create_label_array_for_tile(ctx, label_data, attrib_to_burn=None, layer_idx=0, background_value=255, device=None,
                                label_crs=None):
    """Rasterises the label polygons within the geocontext -> (S, S) uint8 CUDA tensor, S = tilesize + 2 * pad
    (reference :633-689: GDAL MEM raster filled with background_value, RasterizeLayer ALL_TOUCHED with the attribute or 1).

    ctx needs ``tilesize``, ``pad`` and ``geotrans`` (GDAL order) like a DLTile, and ``epsg`` or ``crs`` for labels in another
    CRS.  label_data: a GeoJSON path / dict (read_geojson_layer), or a list of layers / one layer = list of (rings,
    properties).  The layer's CRS is resolved by label_layer_epsg (label_crs, then the GeoJSON ``crs`` member, then
    longitude / latitude detection); longitude / latitude (EPSG:4326) and WGS84 UTM layers are projected into the tile's
    UTM zone on the device before the burn, as RasterizeLayer transforms each geometry into the raster's SRS."""
    size = int(ctx.tilesize) + int(ctx.pad) * 2                 # reference :660
    layer, crs_member = label_data, None
    if isinstance(label_data, (str, bytes, dict)) or hasattr(label_data, "__fspath__"):
        gj = _load_geojson(label_data)
        layer, crs_member = read_geojson_layer(gj), geojson_crs_epsg(gj)
    elif len(label_data) and isinstance(label_data[0], list):   # several layers: GetLayerByIndex(layer_idx), :668
        layer = label_data[layer_idx]
    gt = [float(v) for v in ctx.geotrans]
    if gt[2] != 0.0 or gt[4] != 0.0:
        raise B2Error("create_label_array_for_tile: rotated geotransforms are out of scope (DLTiles are north-up)")
    tile_epsg = _tile_epsg(ctx)
    layer_epsg = label_layer_epsg(tile_epsg, label_crs, crs_member, layer)
    if layer_epsg != tile_epsg:
        layer = _project_layer(layer, layer_epsg, tile_epsg, device)
    inv1, inv5 = 1.0 / gt[1], 1.0 / gt[5]                       # GDALInvGeoTransform for a north-up raster
    inv0, inv3 = -gt[0] * inv1, -gt[3] * inv5
    feats = []
    for rings, props in layer:
        value = int(props[attrib_to_burn]) if attrib_to_burn else 1          # reference :684-687
        px = []
        for r in rings:
            r = np.asarray(r, dtype=np.float64).reshape(-1, 2)
            px.append(np.stack([inv0 + r[:, 0] * inv1, inv3 + r[:, 1] * inv5], axis=1))
        feats.append((px, value))
    return ops.rasterize_polygons(feats, size, background_value, all_touched=True, device=device)


# ------------------------------------------------------------------------------------------------ one training sample
class DLTileJobConfig:
    """What one sample needs (reference :12-102, same attribute names): the tile, the output folder, product(s), dates,
    cloud limit, label data and burn attribute, bands, label nodata value."""

    def __init__(self, dltile, out_folder_base, dl_product, ref_date, labels_data, min_date=None, max_date=None,
                 max_cloud_fraction=None, label_attr=None, label_lyr_num=0, bands="red green blue", label_nodata_value=255):
        self.DLTILE = dltile
        self.OUTFOLDER = out_folder_base
        self.PRODUCT = dl_product
        self.TARGETDATE = ref_date
        self.MIN_DATE = min_date
        self.MAX_DATE = max_date
        self.MAX_CLOUD_FRACTION = max_cloud_fraction
        self.LABEL_DS = labels_data
        self.LABEL_BURN_ATTR = label_attr
        self.LABEL_LYR_NUM = label_lyr_num
        self.BANDS = bands
        self.LABEL_NODATA_VALUE = label_nodata_value


def _tile_epsg(dltile):
    e = getattr(dltile, "epsg", None)
    if e is None:
        crs = str(getattr(dltile, "crs", "") or "")
        e = int(crs.split(":")[1]) if crs.upper().startswith("EPSG:") else 0
    return int(e)


def create_chips_for_tile(job_details, scene_source=None, device=None):
    """Image chip + label chip for one tile job (reference :693-800): pick the compositor as the reference does (:756-770 —
    a list of products -> stack_products_for_tile; max_cloud_fraction == 0 on "sentinel-2:L1C" -> the cloud-masked median;
    anything else -> the nearest-date mosaic), rasterise the labels, write both as tiled LZW GeoTIFFs named after the tile
    key with ':' -> '#' (:749, :778-797), the label with its nodata value.  Returns (job_details, image path, label path),
    or (job_details, None, None) when no image could be made (:772-773)."""
    from . import _geotiff
    dltile = job_details.DLTILE
    product, bands = job_details.PRODUCT, job_details.BANDS
    if isinstance(product, list):
        assert isinstance(bands, list)                                                    # reference :757
        img = stack_products_for_tile(ctx=dltile, products=product, bands_per_product=bands, scene_source=scene_source)
    elif job_details.MAX_CLOUD_FRACTION == 0 and product == "sentinel-2:L1C":
        img = create_cloudmasked_s2_array(ctx=dltile, min_date=job_details.MIN_DATE, max_date=job_details.MAX_DATE, bands=bands,
                                          scene_source=scene_source)
    else:
        img = create_img_array_for_tile(ctx=dltile, product=product, reference_date=job_details.TARGETDATE,
                                        min_date=job_details.MIN_DATE, max_date=job_details.MAX_DATE,
                                        max_cloud_fraction=job_details.MAX_CLOUD_FRACTION, bands=bands, scene_source=scene_source)
    if img is None:
        return (job_details, None, None)
    img_arr = img.data if isinstance(img, MaskedResult) else img      # GDAL writes the masked array's data as it is
    lbl_arr = create_label_array_for_tile(ctx=dltile, label_data=job_details.LABEL_DS, attrib_to_burn=job_details.LABEL_BURN_ATTR,
                                          layer_idx=job_details.LABEL_LYR_NUM, background_value=job_details.LABEL_NODATA_VALUE,
                                          device=device)
    img_file, lbl_file = _geotiff.write_chip_pair(img_arr, lbl_arr, job_details.OUTFOLDER, dltile.key,
                                                  label_ndv=job_details.LABEL_NODATA_VALUE, geotransform=tuple(dltile.geotrans),
                                                  epsg=_tile_epsg(dltile), device=device)
    return (job_details, img_file, lbl_file)
