#!/usr/bin/env python3
"""Fused parse of cfg3-shaped FloatList shards (512 x 512 x 4 uint16 chips stored as packed float32) to normalised
float32 images and one-hot float32 labels: NORM_ONEHOT_F32 against the two-pass route it replaces.

    python tools/parse_float_bench.py [--shards 8] [--recs 32] [--iters 20] [--legs f32_crc,f32_nocrc,two_pass,control]
                                      [--out FILE.jsonl]

Legs, run alternately (one sample of every leg per round), each sample one pass over every device-resident shard:
  * f32_crc / f32_nocrc: parse_table(..., "norm_onehot_f32") with and without data-CRC verification;
  * two_pass: parse_table(..., "raw") with CRC, then ops.normalise_onehot over the copied payloads;
  * control: parse_table(..., "norm_onehot") on bench.py's cfg2 shards (250 u8 records per shard).
The shards together are far larger than the 126 MB L2, so every pass reads them from HBM.  Times are CUDA events;
algorithmic bytes are computed here from the shapes; the fraction is of a device-to-device copy measured in the same
process.  The card's name and power limit are read in the same run and printed on the first line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dl_image_segmentation_b200 import ops  # noqa: E402

S, B, K = 512, 4, 10


def card(dev):
    d = {"device": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        d["power_limit"], d["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:       # the numbers are still worth having; say why the card line is incomplete
        d["power_limit"] = "unread: %s" % e
    return d


def cfg3_shards(dev, n_shards, recs):
    """n_shards shards of recs cfg3 records (uint16 bands, labels 0..K-1 with 2 % nodata 255), built on the device."""
    g = torch.Generator(device=dev)
    g.manual_seed(3003)
    shards = []
    for s in range(n_shards):
        imgs = torch.randint(0, 10047, (recs, S, S, B), dtype=torch.int32, device=dev, generator=g).to(torch.int16).view(torch.uint16)
        labs = torch.randint(0, K, (recs, S, S), dtype=torch.uint8, device=dev, generator=g)
        labs[torch.rand((recs, S, S), device=dev, generator=g) < 0.02] = 255
        items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=2, h=S, w=S, c=B, th=S, tw=S,
                      identifier=b"448#32#10.0#43#%d#%d" % (s, i)) for i in range(recs)]
        buf, _, total = ops.build_records(items, dev)
        shards.append(buf[:total].clone())
        del buf, imgs, labs
    torch.cuda.synchronize(dev)
    return shards


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def summary(xs):
    xs = np.sort(np.asarray(xs))
    return {"median": round(float(np.median(xs)), 4), "min": round(float(xs[0]), 4), "max": round(float(xs[-1]), 4),
            "p10": round(float(np.percentile(xs, 10)), 4), "p90": round(float(np.percentile(xs, 90)), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shards", type=int, default=8)
    ap.add_argument("--recs", type=int, default=32)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--legs", default="f32_crc,f32_nocrc,two_pass,control")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("parse_float_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    legs = args.legs.split(",")
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    head = card(dev)
    head["tiles_per_cta_env"] = os.environ.get("B2_PARSE_TILES_PER_CTA")
    head["lib"] = os.environ.get("B2CHIPS_LIB", "package")

    # device-to-device copy of 1 GiB: the bandwidth the fractions are taken of
    big = torch.empty((1 << 30,), dtype=torch.uint8, device=dev)
    big2 = torch.empty_like(big)
    for _ in range(3):
        big2.copy_(big)
    copy_ms = summary([event_ms(lambda: big2.copy_(big)) for _ in range(10)])
    copy_gbs = (2 << 30) / (copy_ms["median"] / 1e3) / 1e9
    del big, big2
    head.update({"leg": "card+copy", "copy_1GiB_ms": copy_ms, "copy_GB/s": round(copy_gbs, 1)})
    emit(head)

    n, ns = args.recs, args.shards
    shards = cfg3_shards(dev, ns, n)
    tabs = [ops.open_shard_async(s, dev, max_records=n) for s in shards]
    assert all(t.check("cfg3 shard") == n for t in tabs)
    rec_bytes = [int(s.numel()) / n for s in shards]
    rec = float(np.mean(rec_bytes))                          # framed record: header + Example + footer
    mean = ops.to_device(np.array([3000.5, 2800.25, 2500.0, 4000.1], np.float32), dev)
    std = ops.to_device(np.array([1500.0, 1300.3, 1200.0, 2100.7], np.float32), dev)
    img_e, tgt_e = S * S * B, S * S
    out = (torch.empty((n, img_e), dtype=torch.float32, device=dev), torch.empty((n, tgt_e * K), dtype=torch.float32, device=dev))
    raw = (torch.empty((n, img_e * 4), dtype=torch.uint8, device=dev), torch.empty((n, tgt_e * 4), dtype=torch.uint8, device=dev))
    status = torch.empty((n,), dtype=torch.int32, device=dev)
    keep = []

    def f32(verify):
        def run():
            for t in tabs:
                ops.parse_table(t, "norm_onehot_f32", img_e, tgt_e, verify_crc=verify, mean=mean, std=std, num_classes=K,
                                out=out, status=status)
        return run

    def two_pass():
        keep.clear()
        for t in tabs:
            ops.parse_table(t, "raw", img_e * 4, tgt_e * 4, verify_crc=True, out=raw, status=status)
            keep.append(ops.normalise_onehot(raw[0].view(torch.float32).view(n, S, S, B), raw[1].view(torch.float32).view(n, S, S),
                                             mean, std, K, device=dev))

    # the two routes compute the same bits (last shard)
    f32(True)()
    two_pass()
    torch.cuda.synchronize(dev)
    assert not status.any()
    wi, wt = keep[-1]
    same = bool(torch.equal(out[0].view(torch.int32), wi.reshape(n, -1).view(torch.int32)) and torch.equal(out[1], wt.reshape(n, -1)))
    assert same, "NORM_ONEHOT_F32 differs from raw + normalise_onehot"

    fused_b = rec + 4 * img_e + 4 * tgt_e * K
    two_b = (rec + 4 * img_e + 4 * tgt_e) + (4 * img_e + 4 * tgt_e + 4 * img_e + 4 * tgt_e * K)
    crc_b = rec
    runs = {"f32_crc": (f32(True), fused_b), "f32_nocrc": (f32(False), fused_b), "two_pass": (two_pass, two_b)}

    if "control" in legs:
        import bench as Bm
        Bm.N_SHARDS = ns
        c_shards = Bm.make_shards_on_device(dev, 7)
        cn = Bm.RECS_PER_SHARD
        c_tabs = [ops.open_shard_async(s, dev, max_records=cn) for s in c_shards]
        assert all(t.check("cfg2 shard") == cn for t in c_tabs)
        c_mean = ops.to_device(np.array([127.0, 128.0, 126.5], np.float32), dev)
        c_std = ops.to_device(np.array([73.0, 74.0, 72.5], np.float32), dev)
        c_out = (torch.empty((cn, Bm.H * Bm.W * Bm.C), dtype=torch.float32, device=dev),
                 torch.empty((cn, Bm.H * Bm.W * Bm.K), dtype=torch.float32, device=dev))
        c_status = torch.empty((cn,), dtype=torch.int32, device=dev)
        c_rec = float(np.mean([int(s.numel()) / cn for s in c_shards]))

        def control():
            for t in c_tabs:
                ops.parse_table(t, "norm_onehot", Bm.H * Bm.W * Bm.C, Bm.H * Bm.W, verify_crc=True, mean=c_mean, std=c_std,
                                num_classes=Bm.K, out=c_out, status=c_status)
        runs["control"] = (control, None)

    samples = {k: [] for k in legs}
    for it in range(args.warmup + args.iters):
        for k in legs:
            ms = event_ms(runs[k][0])
            if it >= args.warmup:
                samples[k].append(ms)
    assert not status.any()
    if "control" in legs:
        assert not c_status.any()

    for k in legs:
        per_pass = summary(samples[k])
        if k == "control":
            per_shard = {q: round(v / ns, 4) for q, v in per_pass.items()}
            b = c_rec + 4 * Bm.H * Bm.W * Bm.C + 4 * Bm.H * Bm.W * Bm.K
            gbs = b * cn / (per_shard["median"] / 1e3) / 1e9
            emit({"leg": k, "what": "norm_onehot + CRC, cfg2 (256x256x3 u8, K=10), %d shards x %d records" % (ns, cn),
                  "ms_per_%d_records" % cn: per_shard, "algorithmic_bytes_per_record": round(b), "GB/s": round(gbs, 1),
                  "frac_of_copy": round(gbs / copy_gbs, 4), "samples": args.iters})
            continue
        recs = ns * n
        us_rec = per_pass["median"] * 1e3 / recs
        b = runs[k][1]
        gbs = b / (us_rec / 1e6) / 1e9
        d = {"leg": k, "what": "cfg3 (512x512x4 uint16 FloatList, K=%d), %d shards x %d records" % (K, ns, n),
             "ms_per_pass": per_pass, "us_per_record": round(us_rec, 3), "algorithmic_bytes_per_record": round(b),
             "GB/s": round(gbs, 1), "frac_of_copy": round(gbs / copy_gbs, 4), "samples": args.iters}
        if k in ("f32_crc", "f32_nocrc"):
            d["crc_bytes_per_record"] = round(crc_b)
            d["CRCd_GB/s"] = round(crc_b / (us_rec / 1e6) / 1e9, 1) if k == "f32_crc" else None
        emit(d)
    if "f32_crc" in legs and "two_pass" in legs:
        emit({"leg": "ratio", "two_pass_over_f32_crc": round(float(np.median(samples["two_pass"])) / float(np.median(samples["f32_crc"])), 3),
              "outputs_identical": same})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
