#!/usr/bin/env python3
"""The label reprojection kernel (b2_project_points) and what it adds to create_label_array_for_tile.

    python tools/project_bench.py [--vertices 16777216] [--polygons 50000] [--iters 20] [--out FILE.jsonl]

Legs:
  * kernel: `--vertices` lon/lat vertices (zone 43's band, latitudes -80..80) -> EPSG:32643 (forward) and those UTM vertices
    -> EPSG:32644 (inverse + forward in one thread); 16 M vertices are 256 MB in and 256 MB out, more than the 126 MB L2.
    CUDA events around each launch after warm-up; median over --iters, in ns per vertex;
  * drop-in: wall time (host clock, ending in a device synchronise) of create_label_array_for_tile on a cfg3 tile
    (448 px + 2 x 32 pad, 10 m, zone 43N) with `--polygons` small polygons given in lon/lat (label_crs=4326: flatten,
    upload, project, download, then the burn) against the same layer already in the tile's CRS; the two legs alternate.
The card's name and power limit are read in the same run and printed on the first line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dl_image_segmentation_b200 import _descartes_img_chips as dc  # noqa: E402
from dl_image_segmentation_b200 import ops  # noqa: E402


def card(dev):
    d = {"device": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        d["power_limit"], d["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:       # the numbers are still worth having; say why the card line is incomplete
        d["power_limit"] = "unread: %s" % e
    return d


def kernel_ms(xy, src, dst, iters, dev):
    for _ in range(3):
        ops.project_points(xy, src, dst, device=dev)
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.project_points(xy, src, dst, device=dev)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


class Tile:
    key, tilesize, pad, epsg = "448:32:10.0:43:0:0", 448, 32, 32643
    geotrans = (499680.0, 10.0, 0.0, 5300360.0, 0.0, -10.0)


def small_polygons(rng, n, size=512):
    """n star-shaped polygons of 4..10 vertices, 2..12 px across, over the tile (pixel space)."""
    layer = []
    for f in range(n):
        k = int(rng.integers(4, 11))
        ang = np.sort(rng.random(k)) * 2 * np.pi
        rad = rng.uniform(1.0, 6.0, k)
        c = rng.uniform(0, size, 2)
        ring = np.stack([c[0] + rad * np.cos(ang), c[1] + rad * np.sin(ang)], 1)
        layer.append(([np.vstack([ring, ring[:1]])], {"cls": int(rng.integers(0, 10))}))
    return layer


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--vertices", type=int, default=1 << 24)
    ap.add_argument("--polygons", type=int, default=50000)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("project_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = [card(dev)]
    print(json.dumps(lines[0]), flush=True)

    ref = np.load(os.path.join(ROOT, "tests", "golden", "projection.npz"))        # the series-free reference points
    fwd = max(float(np.abs(ops.project_points(ref["fwd_lonlat"][ref["fwd_epsg"] == e], 4326, int(e), device=dev).cpu().numpy()
                           - ref["fwd_utm"][ref["fwd_epsg"] == e]).max()) for e in np.unique(ref["fwd_epsg"]))
    inv = max(float(np.abs(ops.project_points(ref["inv_utm"][ref["inv_epsg"] == e], int(e), 4326, device=dev).cpu().numpy()
                           - ref["inv_lonlat"][ref["inv_epsg"] == e]).max()) for e in np.unique(ref["inv_epsg"]))
    lines.append({"leg": "accuracy", "forward_max_abs_m": fwd, "inverse_max_abs_deg": inv})
    print(json.dumps(lines[-1]), flush=True)

    g = torch.Generator(device=dev)
    g.manual_seed(43)
    n = args.vertices
    ll = torch.stack([72.0 + 6.0 * torch.rand(n, generator=g, device=dev, dtype=torch.float64),
                      -80.0 + 160.0 * torch.rand(n, generator=g, device=dev, dtype=torch.float64)], 1).contiguous()
    utm = ops.project_points(ll, 4326, 32643, device=dev)
    for leg, xy, src, dst in (("forward 4326->32643", ll, 4326, 32643), ("utm->utm 32643->32644", utm, 32643, 32644)):
        ms = kernel_ms(xy, src, dst, args.iters, dev)
        lines.append({"leg": leg, "vertices": n, "ms": round(ms, 4), "ns_per_vertex": round(ms * 1e6 / n, 4),
                      "gbytes_per_s": round(32.0 * n / (ms * 1e-3) / 1e9, 1)})
        print(json.dumps(lines[-1]), flush=True)
    del ll, utm

    rng = np.random.default_rng(50)
    px = small_polygons(rng, args.polygons)
    gt = Tile.geotrans
    to_map = lambda r: np.stack([gt[0] + r[:, 0] * gt[1], gt[3] + r[:, 1] * gt[5]], 1)
    utm_layer = [([to_map(r) for r in rings], p) for rings, p in px]
    flat = ops.project_points(np.concatenate([rs[0] for rs, _ in utm_layer]), 32643, 4326, device=dev).cpu().numpy()
    lonlat_layer, at = [], 0
    for rs, p in utm_layer:
        lonlat_layer.append(([flat[at:at + len(rs[0])]], p))
        at += len(rs[0])
    legs = {"tile_crs": (utm_layer, None), "lonlat": (lonlat_layer, 4326)}
    times = {k: [] for k in legs}
    outs = {}
    for rep in range(6):
        for k, (layer, crs) in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs[k] = dc.create_label_array_for_tile(Tile, layer, attrib_to_burn="cls", device=dev, label_crs=crs)
            torch.cuda.synchronize()
            if rep:                                                   # the first round warms up
                times[k].append(time.perf_counter() - t0)
    differ = int((outs["tile_crs"] != outs["lonlat"]).sum())
    for k in legs:
        lines.append({"leg": "create_label_array_for_tile " + k, "polygons": args.polygons,
                      "vertices": int(sum(len(rs[0]) for rs, _ in legs[k][0])), "ms_median": round(1e3 * float(np.median(times[k])), 2),
                      "ms_min": round(1e3 * min(times[k]), 2)})
        print(json.dumps(lines[-1]), flush=True)
    lines.append({"pixels_that_differ_between_legs": differ})
    print(json.dumps(lines[-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
