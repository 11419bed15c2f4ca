#!/usr/bin/env python3
"""bench.py — headline benchmark: BASELINE.json configs[1]
"parse sharded TFRecords of 256x256x3 uint8 chips -> float32 normalised batches + one-hot labels (10 classes)".

One STEP = one pass of the hot path (frame scan + length-CRC check, Example index, fused data-CRC verify +
cast + per-band normalise + label one-hot) over one batch = 24 shards x 250 records (the 6000-chip dataset
of configs[0]), record = 262 391 B in, 786 432 + 2 621 440 B of float32 out.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = records/s with the shards already resident in HBM;
`e2e` = the same through the public API starting from pinned HOST buffers (H2D of every shard and D2H of
the per-record tables/status inside the timed region); `roofline` = algorithmic bytes of the dominant
kernel / its CUDA-event time vs the measured HBM copy bandwidth; `cpu_baseline` = the oracle restatement
of the reference's CPU path on a bounded sample.  --impl reference times only that CPU path.
--dump-outputs DIR writes a seeded sample of what the last timed step computed (see dump_outputs); the inputs are
generated from fixed seeds, so two builds given the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 256
C = 3
K = 10
N_SHARDS = 24
RECS_PER_SHARD = 250
KEY_FMT = "256:2:1.0:43:%d:%d"          # DLTile-style identifier (_descartes_img_chips.py:749)


def config_dict(n_gpus):
    return {"workload": "cfg2: parse 24 TFRecord shards x 250 records of 256x256x3 u8 chips + 256x256 u8 labels "
                        "-> float32 per-band normalised + one-hot(10), data CRC-32C verified",
            "records_per_step_per_gpu": N_SHARDS * RECS_PER_SHARD, "shards": N_SHARDS, "num_classes": K,
            "l2_policy": "inputs 1.57 GB and outputs 0.85 GB per shard exceed the 126 MB L2; no flush needed",
            "parallelism": "dp%d (shards partitioned per GPU, no collective on the data path)" % n_gpus}


def algorithmic_bytes_per_record(record_bytes):
    return record_bytes + H * W * C * 4 + H * W * K * 4


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self._stop, self.max_mhz = [], set(), threading.Event(), None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            pass
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=1)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ ours
def make_shards_on_device(dev, seed):
    """Synthetic shards built by the product's own writer kernel (tests prove it byte-exact vs the oracle)."""
    import torch

    from dl_image_segmentation_b200 import ops
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    shards = []
    for s in range(N_SHARDS):
        imgs = torch.randint(0, 256, (RECS_PER_SHARD, H, W, C), dtype=torch.uint8, device=dev, generator=g)
        labs = torch.randint(0, K, (RECS_PER_SHARD, H, W), dtype=torch.uint8, device=dev, generator=g)
        nodata = torch.rand((RECS_PER_SHARD, H, W), device=dev, generator=g) < 0.02
        labs[nodata] = 255
        items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=1, h=H, w=W, c=C, th=H, tw=W,
                      identifier=(KEY_FMT % (s, i)).encode()) for i in range(RECS_PER_SHARD)]
        buf, offs, total = ops.build_records(items, dev)
        shards.append(buf[:total].clone())
        del imgs, labs, nodata, buf
    return shards


def run_ours(args, rank, world):
    import torch
    import torch.distributed as dist

    from dl_image_segmentation_b200 import _lib, ops

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        ops.bind_host_to_gpu(local)             # pinned staging memory on the NUMA node next to this rank's GPU
        dist.init_process_group("nccl", device_id=dev)
    ctx = _lib.get_ctx(dev)
    shards = make_shards_on_device(dev, 2002 + rank)
    rec_bytes = shards[0].numel() // RECS_PER_SHARD
    # per-band statistics of the dataset -> mean/std (K4 stats kernel; one tiny allreduce when world > 1)
    si0 = ops.open_shard(shards[0], dev)
    raw_i, _, _ = ops.parse_shard(si0, "raw", verify_crc=False)
    acc = ops.band_stats(raw_i[:, :H * W * C].reshape(-1, C), device=dev)
    if world > 1:
        dist.all_reduce(acc)                      # exact integer counters: identical mean/std on every rank
    mean, std = ops.mean_std_from_stats(ops.stats_to_python(acc))
    mean_d, std_d = ops.to_device(mean, dev), ops.to_device(std, dev)
    del raw_i, si0
    pinned = [s.cpu().pin_memory() for s in shards]
    max_bytes = max(int(s.numel()) for s in shards)
    # the reader's public streaming API: upload (host shards) -> open -> fused parse, no per-shard host sync
    pipe = ops.ShardPipeline("norm_onehot", H * W * C, H * W, max_records=RECS_PER_SHARD, verify_crc=True, mean=mean_d,
                             std=std_d, num_classes=K, device=dev, depth=3, max_shard_bytes=max_bytes)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    kern_events = []
    want = torch.tensor([RECS_PER_SHARD, 0, 0], dtype=torch.int64, device=dev)

    idx014 = torch.tensor([0, 1, 4], dtype=torch.int64, device=dev)

    def make_pass(source):
        """One pass over all shards as a CUDA graph; per shard the consumer folds |records - expected| + scan status +
        bad records into one device-side status word."""
        bad = torch.zeros((), dtype=torch.int64, device=dev)

        def consume(img, tgt, status, table):
            bad.add_((table.hdr_dev.index_select(0, idx014) - want).abs().sum())
            return img, tgt, status, table                      # kept in CapturedPass.results (for --dump-outputs)
        return ops.CapturedPass(pipe, source, consume), bad

    pass_res, bad_res = make_pass(shards)
    pass_e2e, bad_e2e = make_pass(pinned)                       # H2D of every shard inside the graph
    host_status = torch.zeros((), dtype=torch.int64).pin_memory()

    def step_resident():
        pass_res.replay()
        return bad_res

    def step_e2e():
        bad_e2e.zero_()
        pass_e2e.replay()
        host_status.copy_(bad_e2e, non_blocking=True)           # D2H: the job's status word
        torch.cuda.current_stream().synchronize()
        if int(host_status):
            raise RuntimeError("parse status != 0")
        return bad_e2e

    ev_out = (torch.empty((RECS_PER_SHARD, H * W * C), dtype=torch.float32, device=dev),
              torch.empty((RECS_PER_SHARD, H * W * K), dtype=torch.float32, device=dev))

    def step_kernel_events():
        """Un-pipelined pass with CUDA events around every launch of the dominant kernel (same stream)."""
        out, status = ev_out, None
        for s in shards:
            st = ops.open_shard_async(s, dev, max_records=RECS_PER_SHARD)
            a, b = ev(), ev()
            a.record()
            i_, t_, status = ops.parse_table(st, "norm_onehot", H * W * C, H * W, verify_crc=True, mean=mean_d, std=std_d,
                                             num_classes=K, out=out, status=status)
            b.record()
            out = (i_, t_)
            kern_events.append((a, b))
            assert st.check("bench shard") == RECS_PER_SHARD

    own_ms = {}

    def timed(fn, steps, warmup, keep_own=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        last = None
        for _ in range(steps):
            last = fn()
        b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = a.elapsed_time(b)
        if keep_own:
            own_ms["e2e"] = [ms]
        if world > 1:
            if keep_own:                                     # every rank's own time: which rank the host fabric starves
                g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
                dist.all_gather(g, torch.tensor([ms], dtype=torch.float64, device=dev))
                own_ms["e2e"] = [float(x.item()) for x in g]
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, last

    host_sample = [p.numpy().tobytes() for p in pinned[:4]] if rank == 0 and not args.no_cpu_baseline else None
    sampler = ClockSampler(local)
    sampler.start()
    bad_res.zero_()
    ms, bad = timed(step_resident, args.steps, args.warmup)
    clocks = sampler.stop()
    assert int(bad.cpu()) == 0, "parse status != 0"
    if args.dump_outputs and rank == 0:                         # before the e2e pass reuses the pipeline's buffers
        dump_outputs(args.dump_outputs, pass_res.results[-pipe.depth:], idx014)
    launches = pass_res.launches_per_replay * args.steps        # our kernels inside the timed region (graph nodes)
    step_kernel_events()                                    # warm-up of the un-pipelined order
    del kern_events[:]
    step_kernel_events()                                    # per-launch CUDA events of the dominant kernel
    step_kernel_events()
    e2e_steps = args.steps
    ms_e2e, _ = timed(step_e2e, e2e_steps, 3, keep_own=True)

    recs_step = N_SHARDS * RECS_PER_SHARD
    value = world * recs_step * args.steps / (ms / 1e3)
    e2e_value = world * recs_step * e2e_steps / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
    traffic = args.traffic
    if traffic is None:                                     # dram bytes per launch from the committed ncu --set full capture
        try:
            traffic = float(json.load(open(os.path.join(ROOT, "profiles", "r02_parse_traffic.json")))["dram_bytes_per_launch"])
        except Exception:
            traffic = None
    kms = [a.elapsed_time(b) for a, b in kern_events]
    k_avg_ms = sum(kms) / len(kms)
    algo = algorithmic_bytes_per_record(rec_bytes) * RECS_PER_SHARD
    achieved = algo / (k_avg_ms / 1e3) / 1e9
    # inside the timed CUDA-graph step the 24 fused passes run on 3 streams and overlap each other's head and tail, so
    # the per-launch time there is at most ms_per_step / 24 (which also contains the open kernels)
    in_graph_ms = ms / args.steps / N_SHARDS
    h2d = int(sum(p.numel() for p in pinned))
    line = {
        "metric": "chips/sec (parse TFRecord -> normalised float32 tensor + one-hot)", "value": value, "unit": "chips/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8->f32", "data": "synthetic",
        "config": config_dict(world), "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "chips/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 8, "steps": e2e_steps,
                "results": "float32 batches stay on the device (SURVEY 8b: torch.Tensor on CUDA); D2H is the job's status word",
                "per_rank": [{"rank": r, "chips_per_s": recs_step * e2e_steps / (m / 1e3), "h2d_GB/s": h2d * e2e_steps / (m / 1e3) / 1e9}
                             for r, m in enumerate(own_ms["e2e"])],
                "h2d_GB/s_aggregate": world * h2d * e2e_steps / (ms_e2e / 1e3) / 1e9},
        "roofline": {"bound": "hbm", "kernel": "fused_parse_kernel<NORM_ONEHOT> (CRC-32C verify + normalise + one-hot)", "achieved": achieved,
                     "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                     "launch_ms": k_avg_ms, "launch_timing": "CUDA events around each launch, un-pipelined pass on one stream",
                     "algorithmic_bytes_per_launch": algo, "traffic": traffic,
                     "traffic_source": "ncu --set full capture of this kernel, profiles/r02_parse_traffic.json (dram read + write per launch)",
                     "in_graph": {"ms_per_launch_upper_bound": in_graph_ms, "achieved": algo / (in_graph_ms / 1e3) / 1e9,
                                  "frac": algo / (in_graph_ms / 1e3) / 1e9 / peak,
                                  "note": "ms_per_step / 24 launches: inside the timed graph consecutive passes overlap on 3 streams"}},
    }
    if not args.no_other_configs:
        del pass_res, pass_e2e, pipe, pinned, shards, ev_out
        torch.cuda.empty_cache()
        try:
            line["other_configs"] = other_configs(dev) if world == 1 else {}
        except Exception as e:                              # never lose the headline line to a secondary measurement
            line["other_configs"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        for name, fn in (("cfg5_mosaic_1M_chips_strong_scaling", lambda: mosaic_strong(dev, rank, world)),
                         ("cfg1_translate_e2e_png_to_array_records", lambda: translate_e2e(dev, rank, world, "png", True)),
                         ("cfg3_translate_e2e_lzw_geotiff_to_array_records", lambda: translate_e2e(dev, rank, world, "lzw", True)),
                         ("cfg3_translate_e2e_lzw_geotiff_to_raw_records", lambda: translate_e2e(dev, rank, world, "lzw", False))):
            try:
                line["other_configs"][name] = fn()
            except Exception as e:
                line["other_configs"][name] = {"error": repr(e)}
                if world > 1:
                    raise                                   # a rank that drops out of a collective leg hangs the others
            torch.cuda.empty_cache()
    if rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(host_sample, mean, std, budget_s=12.0)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(line))


DUMP_SEED = 2002
DUMP_SAMPLES = 1 << 20                  # per shard and output array: 2 x 3 x 4 MiB = 24 MiB written in all


def dump_outputs(out_dir, results, hdr_fields):
    """Write what the last timed step handed its consumer, so that two builds can be compared output for output.

    A shard's output buffers are recycled `depth` shards later, so after the step the results of the last `depth` shards
    are the ones still on the device.  Their normalised images and one-hot labels (0.85 GB per shard) are sampled at
    DUMP_SAMPLES positions drawn once from DUMP_SEED; the per-record status and the table header (records, scan status,
    records failing the data CRC) are written whole."""
    import torch
    rng = np.random.default_rng(DUMP_SEED)
    dev = results[0][0].device
    picks = [torch.from_numpy(np.sort(rng.choice(results[0][i].numel(), DUMP_SAMPLES, replace=False))).to(dev) for i in (0, 1)]
    arrays = {"image_sample": torch.stack([r[0].reshape(-1)[picks[0]] for r in results]),
              "onehot_sample": torch.stack([r[1].reshape(-1)[picks[1]] for r in results]),
              "record_status": torch.stack([r[2] for r in results]).to(torch.float32),
              "shard_header": torch.stack([r[3].hdr_dev.index_select(0, hdr_fields) for r in results]).to(torch.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def _mosaic_traffic(chips_per_s, peak):
    """DRAM bytes per chip of the mosaic kernel from the committed ncu --set full capture, and the rate they imply."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_mosaic_traffic.json")))
        b = float(t["dram_bytes_per_chip"])
        return {"bytes_per_chip_ncu": b, "GB/s": chips_per_s * b / 1e9, "frac_of_measured_hbm": round(chips_per_s * b / 1e9 / peak, 4),
                "source": "profiles/r02_mosaic_traffic.json (dram__bytes_read + write of one launch / 4096 chips)"}
    except Exception:
        return None


def other_configs(dev):
    """The other configurations of BASELINE.json's compound metric, device-resident kernel rates on this GPU (CUDA
    events, inputs >> L2, same code as tools/kbench.py): cloud-masked median (configs[3]), nearest-date mosaic with
    fused band statistics (configs[4]), chip decode and record build (configs[0] PNG, configs[2] LZW GeoTIFF).
    Reported next to the headline, not part of `value`."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import kbench
    kbench.QUIET = True
    os.environ.setdefault("KB_DECODE_REPS", "64")           # 1024 chip pairs per decode batch
    out = {}

    def keep(d, *keys):
        return {k: d[k] for k in ("ms", "GB/s", "frac_of_measured_hbm") + keys if k in d}
    d = kbench.bench_median(dev, n_tiles=8, iters=16)
    out["cfg4_median_T16_1024x1024x8_u16"] = keep(d, "tiles_per_s", "Gpix_per_s")
    torch.cuda.empty_cache()
    d = kbench.bench_mosaic(dev, pool=256, chips=4096, iters=5, stats=True)
    out["cfg5_mosaic_T32_256x256x4_u16_with_band_stats"] = {
        "ms": d["ms"], "chips_per_s": d["chips_per_s"], "min_touched_GB/s": d["GB/s_min_touched"],
        "frac_of_measured_hbm_min_touched": round(d["GB/s_min_touched"] / kbench.PEAK, 4), "dense_equivalent_GB/s": d["GB/s"],
        "dram_traffic": _mosaic_traffic(d["chips_per_s"], kbench.PEAK),
        "note": "SURVEY 8(d): 331 k chips/s is the dense-definition roofline; the kernel skips filtered / occluded scenes, so the "
                "dense-equivalent rate exceeds HBM bandwidth and the fraction is quoted on the bytes it must touch"}
    torch.cuda.empty_cache()
    for d, name in zip(kbench.bench_build(dev, n_shards=4), ("cfg1_record_build_u8_bytes", "cfg3_record_build_u16_to_floatlist")):
        out[name] = keep(d, "records_per_s")
    torch.cuda.empty_cache()
    d = kbench.bench_decode(dev, "png")
    out["cfg1_png_decode"] = keep(d, "chip_pairs_per_s", "decoded_GB/s")
    d = kbench.bench_decode(dev, "lzw")
    out["cfg3_lzw_geotiff_decode"] = keep(d, "chip_pairs_per_s", "decoded_GB/s")
    d = kbench.bench_jpeg(dev)
    out["cfg1_jpeg_decode"] = keep(d, "chip_pairs_per_s", "decoded_GB/s")
    d = kbench.bench_jpeg_encode(dev)
    out["cfg1_jpeg_encode_png_to_jpg"] = keep(d, "chip_pairs_per_s", "file_MB")
    torch.cuda.empty_cache()
    return out


def _all_max(x, dev, world):
    import torch
    import torch.distributed as dist
    if world == 1:
        return [float(x)]
    g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
    dist.all_gather(g, torch.tensor([x], dtype=torch.float64, device=dev))
    return [float(t.item()) for t in g]


def mosaic_strong(dev, rank, world, chips=1_000_000, batch=4096, pool=256):
    """BASELINE.json configs[4]: nearest-date mosaic with date / cloud filters, T=32, ONE fixed 1M-chip dataset split over
    the ranks by the reference's linspace ranges (strong scaling), per-band statistics fused into the mosaic kernel and
    combined by the path's single collective (all_reduce of exact integer counters) -> mean / std bit-identical for any N."""
    import hashlib

    import torch
    import torch.distributed as dist

    import synthetic as syn
    from dl_image_segmentation_b200 import _lib, ops
    ctx = _lib.get_ctx(dev)
    T, HH, WW, B = 32, 256, 256, 4
    g = torch.Generator(device=dev)
    g.manual_seed(1005)
    stacks = torch.randint(0, 10001, (pool, T, HH, WW, B), dtype=torch.int32, device=dev, generator=g).to(torch.int16).view(torch.uint16)
    coarse = torch.rand((pool * T, 1, 16, 16), device=dev, generator=g)
    valids = (torch.nn.functional.interpolate(coarse, size=(HH, WW), mode="bilinear") > 0.15).to(torch.uint8).reshape(pool, T, HH, WW)
    day = torch.sort(torch.randint(0, 730, (chips, T), dtype=torch.int32, device=dev, generator=g), dim=1).values.contiguous()
    cf = torch.rand((chips, T), dtype=torch.float32, device=dev, generator=g)
    spacing = np.linspace(0, chips, world + 1).astype(int)
    lo, hi = int(spacing[rank]), int(spacing[rank + 1])
    sp_all = torch.tensor([stacks[c].data_ptr() for c in range(pool)], dtype=torch.int64, device=dev)
    vp_all = torch.tensor([valids[c].data_ptr() for c in range(pool)], dtype=torch.int64, device=dev)
    out = torch.empty((batch, HH, WW, B), dtype=torch.uint16, device=dev)
    mask = torch.empty((batch, HH, WW), dtype=torch.uint8, device=dev)
    nel = torch.empty((batch,), dtype=torch.int32, device=dev)
    acc = torch.zeros((B, 4), dtype=torch.int64, device=dev)
    none_count = torch.zeros((), dtype=torch.int64, device=dev)
    f = syn.CFG5_FILTER
    l0 = ctx.launches

    def run(c0, c1):
        n = c1 - c0
        idx = torch.arange(c0, c1, device=dev) % pool
        sp, vp = sp_all[idx], vp_all[idx]
        _lib.check(_lib.lib().b2_nearest_date_mosaic(ctx.handle, _lib.ptr(sp), _lib.ptr(vp), _lib.ptr(day[c0:c1]), _lib.ptr(cf[c0:c1]),
                                                     f["ref_day"], f["min_day"], f["max_day"], f["max_cf"], n, T, HH, WW, B, 2,
                                                     _lib.ptr(out), _lib.ptr(mask), None, _lib.ptr(nel), _lib.ptr(acc), ctx.stream()))
        none_count.add_((nel[:n] == 0).sum())
    for _ in range(3):
        run(lo, min(hi, lo + batch))                            # warm-up
    acc.zero_()
    none_count.zero_()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launches
    a.record()
    for c0 in range(lo, hi, batch):
        run(c0, min(hi, c0 + batch))
    if world > 1:
        dist.all_reduce(acc)                                    # the single collective of the path
        dist.all_reduce(none_count)
    b.record()
    torch.cuda.synchronize()
    launches = ctx.launches - l0
    per_rank = _all_max(a.elapsed_time(b), dev, world)
    ms = max(per_rank)
    stats = ops.stats_to_python(acc)
    mean, std = ops.mean_std_from_stats(stats)
    dense = chips * (T * HH * WW * B * 2 + T * HH * WW + HH * WW * B * 2 + HH * WW)
    del stacks, valids, day, cf, out, mask
    return {"chips": chips, "scaling": "strong", "n_gpus": world, "ms": ms, "chips_per_s": chips / ms * 1e3, "per_rank_ms": per_rank,
            "dense_equivalent_GB/s_per_gpu": dense / world / ms / 1e6, "mosaic_kernel_launches_this_rank": int(launches),
            "collectives": 0 if world == 1 else 2, "chips_without_any_eligible_scene": int(none_count.item()),
            "band_mean": [float(x) for x in mean], "band_std": [float(x) for x in std],
            "band_stats_sha256": hashlib.sha256(repr(stats).encode()).hexdigest()[:16],
            "note": "band_stats_sha256 (exact integer n, sum, sum of squares per band) must be equal for every n_gpus"}


TRANSLATE = {"png": dict(pairs_per_gpu=6000, shards_per_gpu=24, ext="png", cpu_pairs=1500),
             "lzw": dict(pairs_per_gpu=512, shards_per_gpu=8, ext="tif", cpu_pairs=256)}


def _make_chip_files(kind, root, lo, hi, distinct=64):
    """Files lo..hi of the synthetic chip folder: `distinct` different chips encoded once (by whoever gets there first),
    the rest copies under fresh DLTile keys."""
    import shutil

    import synthetic as syn
    ext = TRANSLATE[kind]["ext"]
    os.makedirs(os.path.join(root, "images"), exist_ok=True)
    os.makedirs(os.path.join(root, "labels"), exist_ok=True)

    def name(i):
        return ("256#2#1.0#43#%d#%d.%s" if kind == "png" else "448#32#10.0#43#%d#%d.%s") % (i // 1000, i % 1000, ext)

    def encode(i):
        if kind == "png":
            img, lab, _ = syn.cfg1_chip(i)
            return syn.png_bytes(img), syn.png_bytes(lab)
        img, lab, _ = syn.cfg3_chip(i)
        return syn.tiff_bytes(img, tile=256), syn.tiff_bytes(lab, tile=256, nodata=255)
    nbytes = 0
    for i in range(lo, hi):
        src = i % distinct
        for sub in ("images", "labels"):
            dst = os.path.join(root, sub, name(i))
            if i < distinct:
                continue
            shutil.copyfile(os.path.join(root, "_distinct", sub, "%d.%s" % (src, ext)), dst)
            nbytes += os.path.getsize(dst)
    return nbytes, name, encode


def translate_e2e(dev, rank, world, kind, store_as_array):
    """BASELINE.json configs[0] / configs[2] end to end through the drop-in `images_to_tfrecords_mp`: chip files on /dev/shm
    -> decode -> Example + framing + CRC-32C -> shard files, one process per GPU (worker p = rank p, the reference's
    partition), weak scaling (pairs_per_gpu per rank).  Rank 0's shards are compared byte for byte with the CPU
    restatement of the reference's worker loop, which is timed on processes over all host cores beside it."""
    import contextlib
    import io
    import shutil
    import tempfile

    import torch
    import torch.distributed as dist
    from joblib import Parallel, delayed

    import dl_image_segmentation_b200 as pkg
    import synthetic as syn
    cfg = TRANSLATE[kind]
    n, shards, ext = cfg["pairs_per_gpu"] * world, cfg["shards_per_gpu"] * world, cfg["ext"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    root = os.path.join(base, "b2bench_%s_%d" % (kind, int(os.environ.get("MASTER_PORT", "0")) or os.getppid()))
    distinct = 64
    cores = os.cpu_count() or 1
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
        for sub in ("images", "labels", "_distinct/images", "_distinct/labels"):
            os.makedirs(os.path.join(root, sub))
        _, name, encode = _make_chip_files(kind, root, 0, 0)

        def one(i):
            a, b = encode(i)
            for sub, blob in (("images", a), ("labels", b)):
                open(os.path.join(root, "_distinct", sub, "%d.%s" % (i, ext)), "wb").write(blob)
                open(os.path.join(root, sub, name(i)), "wb").write(blob)
            return len(a) + len(b)
        first = sum(Parallel(n_jobs=min(cores, 16))(delayed(one)(i) for i in range(distinct)))
    if world > 1:
        dist.barrier()
    lo, hi = np.linspace(0, n, world + 1).astype(int)[rank:rank + 2]
    copied, _, _ = _make_chip_files(kind, root, int(lo), int(hi), distinct)
    if world > 1:
        dist.barrier()
    in_bytes = sum(os.path.getsize(os.path.join(root, sub, f)) for sub in ("images", "labels") for f in os.listdir(os.path.join(root, sub))) \
        if rank == 0 else 0
    from dl_image_segmentation_b200 import _lib
    ctx = _lib.get_ctx(dev)
    out = os.path.join(root, "out")
    warm = os.path.join(root, "warm")

    def job(dst):
        with contextlib.redirect_stdout(io.StringIO()):
            pkg.images_to_tfrecords_mp("bench", root, dst, shards, num_proc=world, file_ext=ext, store_as_array=store_as_array)
        torch.cuda.synchronize()
    job(warm)                                                   # warm-up: contexts, pinned buffers, page cache
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(warm, ignore_errors=True)
    if world > 1:
        dist.barrier()
    l0 = ctx.launches
    t0 = time.time()
    job(out)
    own = time.time() - t0
    launches = ctx.launches - l0
    per_rank = _all_max(own, dev, world)
    secs = max(per_rank)
    res = {"pairs": n, "pairs_per_gpu": cfg["pairs_per_gpu"], "shards": shards, "scaling": "weak", "n_gpus": world,
           "store_as_array": store_as_array, "seconds": secs, "pairs_per_s": n / secs, "per_rank_s": per_rank,
           "kernel_launches_this_rank": int(launches), "timing": "wall clock around the whole job incl. file reads and shard "
           "writes (host I/O is part of the metric), max over ranks, after one warm-up job", "files_on": base}
    if rank == 0:
        res["input_MB"] = in_bytes / 1e6
        res["output_MB"] = sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out)) / 1e6
        # CPU restatement of the reference's worker loop on processes (joblib/loky like the reference), on the first
        # cpu_pairs files of the shuffled list = a prefix of worker 0's range -> same records as the head of rank 0's shards
        from oracle import partition as opart
        from oracle import tfrecord as otfr
        from oracle import translate as otr
        n_cpu = min(cfg["cpu_pairs"], cfg["pairs_per_gpu"])
        procs = min(cores, 32)
        cpu_out = os.path.join(root, "cpu")
        t0 = time.time()
        otr.images_to_tfrecords("cpu", root, cpu_out, procs, num_proc=procs, file_ext=ext, store_as_array=store_as_array,
                                n_jobs=procs, limit=n_cpu)
        cpu_s = time.time() - t0
        res["cpu_reference_restatement"] = {"pairs": n_cpu, "processes": procs, "cores": cores, "seconds": cpu_s,
                                            "pairs_per_s": n_cpu / cpu_s, "kind": "port"}
        want = b"".join(open(os.path.join(cpu_out, opart.shard_name("cpu", k, procs)), "rb").read() for k in range(procs))
        got = b""
        k = 0
        while len(got) < len(want):
            got += open(os.path.join(out, opart.shard_name("bench", k, shards)), "rb").read()
            k += 1
        res["byte_identical_with_cpu_restatement"] = bool(got[:len(want)] == want)
        res["records_compared"] = len(otfr.scan(want, verify=False)[0])
        if world > 1:
            # the other end of the partition too: the head of the LAST rank's first shard, record by record
            imgs, lbls = opart.find_image_files(root, ext)
            plan = opart.shard_plan(len(imgs), shards, world)
            sh, lo, hi = plan[(world - 1) * cfg["shards_per_gpu"]]
            k = min(32, hi - lo)
            want2 = b"".join(otfr.frame(otr.build_record(imgs[i], lbls[i], True, store_as_array)) for i in range(lo, lo + k))
            with open(os.path.join(out, opart.shard_name("bench", sh, shards)), "rb") as f:
                got2 = f.read(len(want2))
            res["last_rank_first_shard_head_identical"] = bool(got2 == want2)
            res["records_compared"] += k
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
    return res


# ------------------------------------------------------------------------------------------------ CPU arm (oracle)
def _parse_file(path, mean, std):
    """One tf.data worker's share: read a piece of a shard file, verify CRCs, parse, cast + normalise + one-hot."""
    from oracle import translate
    with open(path, "rb") as f:
        buf = f.read()
    imgs, hots = translate.parse_shard_bytes(buf, mean, std, K, verify=True)
    return int(imgs.shape[0])


def _shard_pieces(host_shards, chunk, tmpdir):
    """Cut shards into files of `chunk` whole records (the reference maps per record over 8 parallel calls; a piece per
    task keeps every process busy without pickling megabytes per call)."""
    from oracle import tfrecord as otfr
    paths = []
    for si, buf in enumerate(host_shards):
        offs, lens = otfr.scan(buf, verify=False)
        for i in range(0, len(offs), chunk):
            j = min(i + chunk, len(offs)) - 1
            p = os.path.join(tmpdir, "piece-%03d-%05d" % (si, i))
            with open(p, "wb") as f:
                f.write(buf[int(offs[i]) - 12:int(offs[j] + lens[j]) + 4])
            paths.append((p, j - i + 1))
    return paths


def _cpu_tmpdir():
    import tempfile
    return tempfile.mkdtemp(prefix="b2cpu_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)


def cpu_baseline(host_shards, mean, std, budget_s=12.0, chunk=25):
    """Oracle restatement of TFRecordDataset(files).map(parse_fn, num_parallel_calls) + cast / normalise / one-hot on
    the host cores: one OS process per core (no GIL between workers), shard pieces read from files."""
    import shutil

    from joblib import Parallel, delayed
    cores = os.cpu_count() or 1
    tmp = _cpu_tmpdir()
    try:
        pieces = _shard_pieces(host_shards, chunk, tmp)
        done = 0
        with Parallel(n_jobs=cores) as par:
            par(delayed(_parse_file)(p, mean, std) for p, _ in pieces[:2 * cores])     # warm-up: workers start, imports
            t0 = time.time()
            i = 0
            while time.time() - t0 < budget_s:
                batch = [pieces[(i + k) % len(pieces)][0] for k in range(8 * cores)]
                done += sum(par(delayed(_parse_file)(p, mean, std) for p in batch))
                i += len(batch)
            dt = time.time() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return {"value": done / dt, "unit": "chips/s", "cores": cores, "kind": "port",
            "sample": "%d records (4 of the shards, cycled) over %d worker processes (reference: dataset.map(parse_fn, 8)), %.1f s; "
                      "restatement because TensorFlow is not installable" % (done, cores, dt)}


def make_shards_on_host(seed, n_shards):
    from oracle import example_proto as oep
    from oracle import tfrecord as otfr
    rng = np.random.default_rng(seed)
    shards = []
    for s in range(n_shards):
        parts = []
        for i in range(RECS_PER_SHARD):
            img = rng.integers(0, 256, (H, W, C), dtype=np.uint8)
            lab = rng.integers(0, K, (H, W), dtype=np.uint8)
            lab[rng.random((H, W)) < 0.02] = 255
            parts.append(otfr.frame(oep.convert_to_example(img, lab, H, W, C, H, W, KEY_FMT % (s, i)).SerializeToString()))
        shards.append(b"".join(parts))
    return shards


def run_reference(args, rank, world):
    """The reference's CPU path (oracle restatement) on the host cores, one process per core; rank 0 only."""
    if rank != 0:
        return
    import shutil

    from joblib import Parallel, delayed
    cores = os.cpu_count() or 1
    shards = make_shards_on_host(2002, 4)
    mean = np.array([127.5, 127.5, 127.5], np.float32)
    std = np.array([73.9, 73.9, 73.9], np.float32)
    tmp = _cpu_tmpdir()
    try:
        pieces = _shard_pieces(shards, 25, tmp)                  # 40 pieces of 25 records
        n_step = sum(n for _, n in pieces)                       # one step = 4 shards = 1000 records (bounded sample of the 6000)
        with Parallel(n_jobs=cores) as par:
            for _ in range(max(1, args.warmup)):
                par(delayed(_parse_file)(p, mean, std) for p, _ in pieces)
            t0 = time.time()
            for _ in range(args.steps):
                got = sum(par(delayed(_parse_file)(p, mean, std) for p, _ in pieces))
                assert got == n_step
            dt = time.time() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    value = n_step * args.steps / dt
    sample = ("each step parses 4 shards (%d records) of the %d-record batch over %d worker processes; restatement of "
              "TFRecordDataset.map(parse_fn)+normalise+one-hot (TensorFlow not installable)" % (n_step, N_SHARDS * RECS_PER_SHARD, cores))
    line = {"impl": "reference", "metric": "chips/sec (parse TFRecord -> normalised float32 tensor + one-hot)",
            "value": value, "unit": "chips/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8->f32", "data": "synthetic", "config": config_dict(world),
            "cpu_baseline": {"value": value, "unit": "chips/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "chips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the secondary per-config kernel rates (N=1 only)")
    ap.add_argument("--traffic", type=float, default=None, help="dram bytes per launch from an ncu --set full capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
