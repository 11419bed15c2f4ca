#!/usr/bin/env python3
"""Per-band statistics and label histograms straight from the shards (the fused parse's STATS / STATS_F32 sinks) against
the CRC-only pass over the same shards and against the two-pass route they replace.

    python tools/parse_stats_bench.py [--iters 20] [--out FILE.jsonl]

Legs, run alternately (one sample of every leg per round), each sample one pass over every device-resident shard:
  * cfg2 (bench.py's shards: 24 x 250 records of 256x256x3 uint8 + labels, built as bench.py builds them):
    stats_crc / stats_nocrc (parse_table "stats" with and without data-CRC verification), none_crc (parse_table "none":
    the CRC alone), two_pass (parse_table "raw" without CRC, then band_stats over the copied images: bench.py's route);
  * cfg3 (8 x 32 records of 512x512x4 uint16 as packed FloatList, K = 10 labels with 2 % nodata 255):
    stats_f32_crc / stats_f32_nocrc / none_crc;
  * tail: 4736 records of 8x8x3 uint8, one 8 KiB tile each, so that every one of the grid's CTAs runs and flushes its
    counters while the data work is negligible: "stats" minus "none" bounds the cost of the exit flush from above.
The cfg2 and cfg3 shards are each larger than the 126 MB L2, so every pass reads them from HBM.  Times are CUDA events;
bytes read are the shards' sizes; the fraction is of a device-to-device copy measured in the same process.  The card's
name and power limit are read in the same run and printed on the first line.
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

import bench as Bm  # noqa: E402
from dl_image_segmentation_b200 import ops  # noqa: E402

S3, B3, K3 = 512, 4, 10


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
    g = torch.Generator(device=dev)
    g.manual_seed(3003)
    shards = []
    for s in range(n_shards):
        imgs = torch.randint(0, 10047, (recs, S3, S3, B3), dtype=torch.int32, device=dev, generator=g).to(torch.int16).view(torch.uint16)
        labs = torch.randint(0, K3, (recs, S3, S3), dtype=torch.uint8, device=dev, generator=g)
        labs[torch.rand((recs, S3, S3), device=dev, generator=g) < 0.02] = 255
        items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=2, h=S3, w=S3, c=B3, th=S3, tw=S3,
                      identifier=b"448#32#10.0#43#%d#%d" % (s, i)) for i in range(recs)]
        buf, _, total = ops.build_records(items, dev)
        shards.append(buf[:total].clone())
        del buf, imgs, labs
    return shards


def tiny_shard(dev, n):
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    imgs = torch.randint(0, 256, (n, 8, 8, 3), dtype=torch.uint8, device=dev, generator=g)
    labs = torch.randint(0, 10, (n, 8, 8), dtype=torch.uint8, device=dev, generator=g)
    items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=1, h=8, w=8, c=3, th=8, tw=8,
                  identifier=b"t%d" % i) for i in range(n)]
    buf, _, total = ops.build_records(items, dev)
    return buf[:total].clone()


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
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("parse_stats_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    lines = []

    def emit(d):
        lines.append(d)
        print(json.dumps(d), flush=True)

    head = card(dev)
    big = torch.empty((1 << 30,), dtype=torch.uint8, device=dev)
    big2 = torch.empty_like(big)
    for _ in range(3):
        big2.copy_(big)
    copy_ms = summary([event_ms(lambda: big2.copy_(big)) for _ in range(10)])
    copy_gbs = (2 << 30) / (copy_ms["median"] / 1e3) / 1e9
    del big, big2
    head.update({"leg": "card+copy", "copy_1GiB_ms": copy_ms, "copy_GB/s": round(copy_gbs, 1)})
    emit(head)

    # ---- cfg2
    c2 = Bm.make_shards_on_device(dev, 2002)
    n2, C2 = Bm.RECS_PER_SHARD, Bm.C
    img2 = Bm.H * Bm.W * C2
    t2 = [ops.open_shard_async(s, dev, max_records=n2) for s in c2]
    assert all(t.check("cfg2 shard") == n2 for t in t2)
    acc2 = torch.zeros((C2, 5), dtype=torch.int64, device=dev)
    hist2 = torch.zeros((257,), dtype=torch.int64, device=dev)
    raw2 = (torch.empty((n2, img2), dtype=torch.uint8, device=dev), torch.empty((n2, Bm.H * Bm.W), dtype=torch.uint8, device=dev))
    bacc2 = torch.zeros((C2, 4), dtype=torch.int64, device=dev)
    status = torch.zeros((max(n2, 4736),), dtype=torch.int32, device=dev)

    def stats_pass(tabs, mode, C, out, verify):
        def run():
            for t in tabs:
                ops.parse_table(t, mode, verify_crc=verify, channels=C, out=out, status=status)
        return run

    def none_pass(tabs):
        def run():
            for t in tabs:
                ops.parse_table(t, "none", verify_crc=True, status=status)
        return run

    def two_pass():
        for t in t2:
            ops.parse_table(t, "raw", img2, Bm.H * Bm.W, verify_crc=False, out=raw2, status=status)
            ops.band_stats(raw2[0].reshape(-1, C2), acc=bacc2, device=dev)

    # the two routes count the same (one pass each, from zero)
    stats_pass(t2, "stats", C2, (acc2, hist2), True)()
    two_pass()
    a = acc2.cpu().numpy().view(np.uint64)
    same = [(int(r[0]), int(r[1]), int(r[2]) + 65536 * int(r[3])) for r in a] == ops.stats_to_python(bacc2)
    assert same, "STATS differs from raw + band_stats"

    # ---- cfg3
    c3 = cfg3_shards(dev, 8, 32)
    t3 = [ops.open_shard_async(s, dev, max_records=32) for s in c3]
    assert all(t.check("cfg3 shard") == 32 for t in t3)
    acc3 = torch.zeros((B3, 5), dtype=torch.int64, device=dev)
    hist3 = torch.zeros((257,), dtype=torch.int64, device=dev)

    # ---- exit tail
    tiny = tiny_shard(dev, 4736)
    tt = [ops.open_shard_async(tiny, dev, max_records=4736)]
    assert tt[0].check("tiny shard") == 4736
    acct = torch.zeros((3, 5), dtype=torch.int64, device=dev)
    histt = torch.zeros((257,), dtype=torch.int64, device=dev)

    runs = {
        "cfg2_stats_crc": stats_pass(t2, "stats", C2, (acc2, hist2), True),
        "cfg2_stats_nocrc": stats_pass(t2, "stats", C2, (acc2, hist2), False),
        "cfg2_none_crc": none_pass(t2),
        "cfg2_two_pass": two_pass,
        "cfg3_stats_f32_crc": stats_pass(t3, "stats_f32", B3, (acc3, hist3), True),
        "cfg3_stats_f32_nocrc": stats_pass(t3, "stats_f32", B3, (acc3, hist3), False),
        "cfg3_none_crc": none_pass(t3),
        "tail_stats": stats_pass(tt, "stats", 3, (acct, histt), True),
        "tail_none": none_pass(tt),
    }
    samples = {k: [] for k in runs}
    for it in range(args.warmup + args.iters):
        for k, fn in runs.items():
            ms = event_ms(fn)
            if it >= args.warmup:
                samples[k].append(ms)
    torch.cuda.synchronize(dev)
    assert not status.any()

    shard_bytes = {"cfg2": sum(int(s.numel()) for s in c2), "cfg3": sum(int(s.numel()) for s in c3)}
    recs = {"cfg2": len(c2) * n2, "cfg3": len(c3) * 32}
    med = {k: float(np.median(v)) for k, v in samples.items()}
    for k, v in samples.items():
        cfg = k.split("_")[0]
        d = {"leg": k, "ms_per_pass": summary(v), "samples": args.iters}
        if cfg in recs:
            b = shard_bytes[cfg] + (0 if k != "cfg2_two_pass" else recs[cfg] * (Bm.H * Bm.W * (C2 + 1) + img2))
            d.update({"us_per_record": round(med[k] * 1e3 / recs[cfg], 3), "shard_bytes_per_record": round(shard_bytes[cfg] / recs[cfg]),
                      "bytes_moved_per_record": round(b / recs[cfg]), "TB/s_read": round(shard_bytes[cfg] / (med[k] / 1e3) / 1e12, 3),
                      "frac_of_copy": round(shard_bytes[cfg] / (med[k] / 1e3) / 1e9 / copy_gbs, 4)})
        emit(d)
    emit({"leg": "ratios",
          "cfg2_stats_crc_over_none_crc": round(med["cfg2_stats_crc"] / med["cfg2_none_crc"], 3),
          "cfg3_stats_f32_crc_over_none_crc": round(med["cfg3_stats_f32_crc"] / med["cfg3_none_crc"], 3),
          "cfg2_two_pass_over_stats_nocrc": round(med["cfg2_two_pass"] / med["cfg2_stats_nocrc"], 3),
          "tail_stats_minus_none_us": round((med["tail_stats"] - med["tail_none"]) * 1e3, 2),
          "stats_equal_raw_band_stats": same})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
