"""The fused parse's statistics sinks: STATS (uint8 BytesList records) and STATS_F32 (packed float32 FloatList records)
count exact per-band image statistics and a 257-bin label histogram in the pass that verifies the CRC.

Every comparison is exact integer equality with the references below (Python ints over the records whose status is 0,
bincount-style bins), and every case runs through the uniform tile map (parse_shard) and the opened-table map
(parse_table, what ShardPipeline and shard_stats run).  Covers band counts on every branch of the band stride, payloads
starting at every residue mod 16, payloads straddling tiles, a record past 2048 CRC tiles, empty and one-element
payloads, all 256 byte labels, constant labels (the warp-aggregated bins), float labels without a bin, excluded image
values, per-record statuses, accumulation across calls and streams, NULL outputs, agreement with raw + band_stats on
full-size cfg2 records, misuse, and which kernel each mode launches.

The references need no GPU; test_reference_* check them against the oracle.
"""
import ctypes
import functools
import json

import numpy as np
import pytest

from _sink_refs import _record
from oracle import example_proto as oep
from oracle import normalise as onorm
from oracle import tfrecord as otfr


# ------------------------------------------------------------------------------------------------ references (CPU)
def ref_band_stats(imgs, C):
    """[(n, sum x, sum x^2, excluded)] per band over (..., C) images, as exact Python ints.  Float values count when they
    are integers in [-2^16, 2^16); any other value (NaN, +-inf, non-integral, out of range) is excluded."""
    out = [[0, 0, 0, 0] for _ in range(C)]
    for img in imgs:
        x = np.asarray(img).reshape(-1, C)
        for c in range(C):
            col = x[:, c]
            if col.dtype.kind == "f":
                f = col.astype(np.float64)
                with np.errstate(invalid="ignore"):
                    ok = (f >= -65536) & (f < 65536) & (f == np.floor(f))
                out[c][3] += int((~ok).sum())
                col = f[ok]
            v = col.astype(np.int64)            # |x| <= 2^16 and fewer than 2^30 values: int64 sums are exact
            out[c][0] += int(v.size)
            out[c][1] += int(v.sum())
            out[c][2] += int((v * v).sum())
    return [tuple(r) for r in out]


def ref_hist(labels):
    """257 bins: bin v counts labels equal to v in 0..255 (-0.0 is 0), bin 256 every other label."""
    bins = [0] * 257
    for lab in labels:
        f = np.asarray(lab).reshape(-1).astype(np.float64)
        with np.errstate(invalid="ignore"):
            ok = (f >= 0) & (f <= 255) & (f == np.floor(f))
        for v, k in enumerate(np.bincount(f[ok].astype(np.int64), minlength=256)):
            bins[v] += int(k)
        bins[256] += int((~ok).sum())
    return bins


def got_stats(acc, hist):
    """Device counters -> ([(n, sum x, sum x^2, excluded)], 257 bins) as Python ints."""
    out = None
    if acc is not None:
        a = acc.cpu().numpy().view(np.uint64)
        out = [(int(r[0]), int(r[1]) - (1 << 64) if int(r[1]) >> 63 else int(r[1]), int(r[2]) + 65536 * int(r[3]), int(r[4]))
               for r in a]
    return out, (None if hist is None else [int(v) for v in hist.cpu().numpy().view(np.uint64)])


@pytest.mark.parametrize("dtype", ("uint8", "uint16"))
def test_reference_matches_oracle_band_stats(dtype):
    rng = np.random.default_rng(5)
    info = np.iinfo(dtype)
    imgs = [rng.integers(0, info.max + 1, (h, w, 3)).astype(dtype) for h, w in ((7, 9), (1, 1), (40, 33))]
    imgs.append(np.full((5, 5, 3), info.max, dtype))
    want = onorm.band_stats(np.concatenate([i.reshape(-1, 3) for i in imgs]))
    assert [r[:3] for r in ref_band_stats(imgs, 3)] == [tuple(int(v) for v in w) for w in want]
    assert all(r[3] == 0 for r in ref_band_stats(imgs, 3))


def test_reference_hist_and_exclusions():
    lab = np.array([-0.0, 0.0, 0.5, -1.0, 255.0, 256.0, np.nan, np.inf, -np.inf, 1e9, 3.0], np.float32)
    h = ref_hist([lab])
    assert h[0] == 2 and h[255] == 1 and h[3] == 1 and h[256] == 7 and sum(h) == lab.size
    img = np.array([1.0, 1.5, np.nan, np.inf, -np.inf, 65536.0, -65537.0, -65536.0, 65535.0], np.float32).reshape(-1, 1)
    assert ref_band_stats([img], 1) == [(3, 0, 1 + 65536 ** 2 + 65535 ** 2, 6)]


# ------------------------------------------------------------------------------------------------ shard fixtures
BANDS = (1, 2, 3, 4, 5, 7, 8, 13, 16, 33, 64)
N_REC = 41
SHAPES = ((1, 1), (1, 7), (3, 5), (29, 31), (32, 32), (0, 5))
BIG = {6: (96, 96), 19: (20, 1100), 30: (64, 64)}
F_LABELS = np.array([-0.0, 0.5, -1.0, 255.0, 256.0, np.nan, np.inf, -np.inf, 1e9, 0.0, 7.0], np.float32)


def _chip(rng, h, w, C, dtype, i):
    """Image of dtype (u8 / u16 / i16 values; float32 storage for FloatList records is the writer's) and labels: random
    bytes, or one constant value every fourth record."""
    if dtype == "uint8":
        img = rng.integers(0, 256, (h, w, C)).astype(np.uint8)
    else:
        info = np.iinfo(dtype)
        img = rng.integers(info.min, info.max + 1, (h, w, C)).astype(dtype)
        img.reshape(-1)[:2] = np.array([info.min, info.max], dtype)[:min(img.size, 2)]
    if i % 4 == 3:
        img[:] = img.reshape(-1)[0] if img.size else 0                  # an image of one value
        lab = np.full((h, w), rng.integers(0, 256), np.uint8)           # a record of one label
    else:
        lab = rng.integers(0, 256, (h, w)).astype(np.uint8)
    return img, lab


@functools.lru_cache(maxsize=None)
def _shard(C, dtype):
    """41 records of C bands; identifier lengths 0..40 move the payload starts through every residue mod 16.  uint8
    images go to BytesList records, the others to FloatList records, whose labels then include float specials."""
    rng = np.random.default_rng(100 * C + len(dtype))
    recs, chips = [], []
    for i in range(N_REC):
        h, w = BIG.get(i, SHAPES[i % len(SHAPES)])
        if C >= 33 and i in BIG:
            h, w = 24, 24
        img, lab = _chip(rng, h, w, C, dtype, i)
        if dtype != "uint8":
            lab = lab.astype(np.float32)
            if i % 4 != 3:
                k = min(lab.size, F_LABELS.size)
                lab.reshape(-1)[:k] = rng.permutation(F_LABELS)[:k]
        recs.append(_record(img, lab, bytes(rng.integers(97, 123, i, dtype=np.uint8))))
        chips.append((img, lab))
    return b"".join(recs), chips


class _Opened:
    def __init__(self, shard, chips, dev, max_records=64):
        from dl_image_segmentation_b200 import ops
        self.si = ops.open_shard(shard, dev, max_records=max_records)
        assert self.si.n == len(chips)
        self.chips = chips


@functools.lru_cache(maxsize=None)
def _opened(C, dtype, dev):
    return _Opened(*_shard(C, dtype), dev)


def _stats_both(op, mode, C, verify_crc=True):
    """Yield (name, bands, bins, status) from parse_shard and from parse_table."""
    from dl_image_segmentation_b200 import ops
    n = op.si.n
    acc, hist, st = ops.parse_shard(op.si, mode, verify_crc=verify_crc, channels=C)
    yield ("parse_shard",) + got_stats(acc, hist) + (st[:n].cpu().numpy(),)
    acc, hist, st = ops.parse_table(op.si.table, mode, verify_crc=verify_crc, channels=C)
    stat = st[:n].cpu().numpy()
    assert op.si.table.header()[4] == int((stat != 0).sum())
    yield ("parse_table",) + got_stats(acc, hist) + (stat,)


def _check(op, mode, C, rows=None, want_status=None):
    rows = range(op.si.n) if rows is None else rows
    want_b = ref_band_stats([op.chips[r][0] for r in rows], C)
    want_h = ref_hist([op.chips[r][1] for r in rows])
    for name, bands, bins, stat in _stats_both(op, mode, C):
        if want_status is None:
            assert not stat.any(), (name, np.nonzero(stat)[0])
        else:
            assert list(stat) == want_status, name
        for c in range(C):
            assert bands[c] == want_b[c], (name, "band", c, bands[c], want_b[c])
        assert bins == want_h, (name, [(v, g, w) for v, (g, w) in enumerate(zip(bins, want_h)) if g != w][:5])


# ------------------------------------------------------------------------------------------------ fused parse (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("C", BANDS)
def test_stats_u8_bands(dev, C):
    """STATS: every band count's stride branch and band cycle, every payload residue, tiles straddled, all 256 labels."""
    _check(_opened(C, "uint8", dev), "stats", C)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ("uint8", "uint16", "int16"))
@pytest.mark.parametrize("C", (1, 3, 4, 5, 8, 13))
def test_stats_f32_bands(dev, C, dtype):
    """STATS_F32: u8-, u16- and i16-valued FloatList images (0, 65535, -32768, constant images included) and float
    labels -0.0, 0.5, -1, 255, 256, NaN, +-inf and 1e9."""
    if dtype == "uint8":
        shard, chips = _shard(C, "uint16")
        rng = np.random.default_rng(C)
        chips = [(rng.integers(0, 256, img.shape).astype(np.uint8), lab) for img, lab in chips]
        shard = b"".join(_record(img, lab, bytes(rng.integers(97, 123, i, dtype=np.uint8))) for i, (img, lab) in enumerate(chips))
        op = _Opened(shard, chips, dev)
    else:
        op = _opened(C, dtype, dev)
    _check(op, "stats_f32", C)


@pytest.mark.gpu
def test_stats_excluded_values(dev):
    """Non-integral, NaN, +-inf, 65536 and -65537 image values land in `excluded` of their band; the band's other values
    and the other bands stay exact; shard_stats refuses the shard naming the band and the count."""
    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    rng = np.random.default_rng(3)
    C = 3
    chips = []
    for i in range(6):
        img = rng.integers(-32768, 65536, (9 + i, 11, C)).astype(np.float32)
        bad = np.array([0.5, np.nan, np.inf, -np.inf, 65536.0, -65537.0, 1e30, -0.25], np.float32)
        img[i % 9, :bad.size, 1] = bad
        chips.append((img, rng.integers(0, 5, (9 + i, 11)).astype(np.float32)))
    shard = b"".join(_record(img, lab, b"x" * i) for i, (img, lab) in enumerate(chips))
    op = _Opened(shard, chips, dev)
    want = ref_band_stats([c[0] for c in chips], C)
    assert want[1][3] == 6 * 8 and want[0][3] == want[2][3] == 0
    _check(op, "stats_f32", C)
    with pytest.raises(B2Error, match="band 1 has 48 value"):
        ops.shard_stats([ops.to_device(shard, dev)], C, kind="float", device=dev)


@pytest.mark.gpu
def test_stats_record_past_2048_tiles(dev):
    """A ~23 MB BytesList record (2400 x 2400 x 3) and a ~19 MiB FloatList record (1100 x 1100 x 4 uint16)."""
    rng = np.random.default_rng(2400)
    chips = [(rng.integers(0, 256, (2400, 2400, 3)).astype(np.uint8), rng.integers(0, 256, (2400, 2400)).astype(np.uint8)),
             (rng.integers(0, 256, (9, 7, 3)).astype(np.uint8), rng.integers(0, 256, (9, 7)).astype(np.uint8))]
    op = _Opened(b"".join(_record(img, lab, b"big%d" % i) for i, (img, lab) in enumerate(chips)), chips, dev, max_records=4)
    assert int(op.si.lens_host[0]) > 2048 * 8192
    _check(op, "stats", 3)
    chips = [(rng.integers(0, 65536, (1100, 1100, 4)).astype(np.uint16), rng.integers(0, 12, (1100, 1100)).astype(np.float32)),
             (rng.integers(0, 65536, (9, 7, 4)).astype(np.uint16), rng.integers(0, 12, (9, 7)).astype(np.float32))]
    op = _Opened(b"".join(_record(img, lab, b"big%d" % i) for i, (img, lab) in enumerate(chips)), chips, dev, max_records=4)
    assert int(op.si.lens_host[0]) > 2048 * 8192
    _check(op, "stats_f32", 4)


class _UnpackedFloats:
    """A FloatList feature with one float per tag (field 1, wire type 5) instead of one packed run."""

    def __init__(self, values):
        self.values = np.asarray(values, "<f4")

    def serialize(self):
        return oep._len_field(2, b"".join(b"\x0d" + v.tobytes() for v in self.values))


def _status_shard(rng, C, kind):
    """Good records of `kind` (1 bytes, 2 float) around records the template refuses (status 2)."""
    recs, chips, want = [], [], []
    fdt = "uint8" if kind == 1 else "uint16"

    def chip(h, w, c=C, dt=fdt):
        img, lab = _chip(rng, h, w, c, dt, 0)
        return (img, lab) if dt == "uint8" else (img, lab.astype(np.float32))

    def add(rec, c, s):
        recs.append(rec)
        chips.append(c)
        want.append(s)

    for i, (h, w) in enumerate(((32, 32), (29, 31), (3, 5), (1, 7), (17, 3), (24, 30))):
        c = chip(h, w)
        add(_record(*c, b"good%d" % i), c, 0)
        if i == 0:
            add(_record(*chip(20, 20, C + 1), b"bands"), chip(1, 1), 2)                       # wrong channel count
        elif i == 1:
            other = chip(8, 8, C, "uint16" if kind == 1 else "uint8")                         # the other payload kind
            if kind == 1:
                other = (other[0], other[1].astype(np.float32))
            add(_record(*other, b"kind"), chip(1, 1), 2)
        elif i == 2:
            add(_record(*chip(10, 10), b"img_len", dims=(11, 10, C, 10, 10)), chip(1, 1), 2)  # image/height says 11
        elif i == 3:
            add(_record(*chip(10, 10), b"tgt_len", dims=(10, 10, C, 9, 10)), chip(1, 1), 2)   # target/height says 9
        elif i == 4:
            img, lab = chip(4, 4, C, "uint16")                                                 # unpacked FloatList image
            ex = oep.convert_to_example(img, lab.astype(np.float32), 4, 4, C, 4, 4, b"unpacked")
            ex.features["image/image_data"] = _UnpackedFloats(img.astype(np.float32).ravel())
            add(otfr.frame(ex.SerializeToString()), chip(1, 1), 2)
    return b"".join(recs), chips, want


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("stats", "stats_f32"))
def test_stats_statuses_keep_neighbours_exact(dev, mode):
    """Records the template refuses get status 2 and add nothing; their neighbours stay exact."""
    C = 4
    shard, chips, want = _status_shard(np.random.default_rng(41), C, 1 if mode == "stats" else 2)
    op = _Opened(shard, chips, dev)
    _check(op, mode, C, rows=[r for r, s in enumerate(want) if s == 0], want_status=want)


@pytest.mark.gpu
def test_stats_crc_mismatch_raises(dev):
    """A payload byte flipped after framing: status 1, and shard_stats raises DataLossError."""
    from dl_image_segmentation_b200 import ops
    rng = np.random.default_rng(9)
    chips = [_chip(rng, 32, 32, 3, "uint8", i) for i in range(3)]
    recs = [bytearray(_record(img, lab, b"crc%d" % i)) for i, (img, lab) in enumerate(chips)]
    recs[1][len(recs[1]) // 2] ^= 0x20
    shard = b"".join(bytes(r) for r in recs)
    op = _Opened(shard, chips, dev)
    for name, _, _, stat in _stats_both(op, "stats", 3):
        assert list(stat) == [0, 1, 0], name
    with pytest.raises(ops.DataLossError, match="1 record\\(s\\) of 1 shard\\(s\\) failed the data CRC"):
        ops.shard_stats([ops.to_device(shard, dev)], 3, device=dev)
    bands, hist = ops.shard_stats([ops.to_device(shard, dev)], 3, device=dev, verify_crc=False)   # nothing checked
    assert [b[0] for b in bands] == [3 * 32 * 32] * 3 and sum(hist) == 3 * 32 * 32


# ------------------------------------------------------------------------------------------------ accumulation (GPU)
@pytest.mark.gpu
def test_stats_accumulate_and_null_outputs(dev):
    """Two calls add up; a NULL acc or hist leaves the other exact and the skipped buffer untouched."""
    import torch

    from dl_image_segmentation_b200 import ops
    C = 5
    op = _opened(C, "uint8", dev)
    want_b = ref_band_stats([c[0] for c in op.chips], C)
    want_h = ref_hist([c[1] for c in op.chips])
    acc = torch.zeros((C, 5), dtype=torch.int64, device=dev)
    hist = torch.zeros((257,), dtype=torch.int64, device=dev)
    ops.parse_table(op.si.table, "stats", channels=C, out=(acc, hist))
    ops.parse_shard(op.si, "stats", channels=C, out=(acc, hist))
    bands, bins = got_stats(acc, hist)
    assert bands == [tuple(2 * v for v in r) for r in want_b] and bins == [2 * v for v in want_h]
    for want_img in (False, True):
        acc = torch.full((C, 5), 7, dtype=torch.int64, device=dev)
        hist = torch.full((257,), 7, dtype=torch.int64, device=dev)
        ops.parse_table(op.si.table, "stats", channels=C, out=(acc, hist), want_img=want_img, want_tgt=not want_img)
        if want_img:
            acc -= 7
            assert got_stats(acc, None)[0] == want_b and bool((hist == 7).all())
        else:
            hist -= 7
            assert got_stats(None, hist)[1] == want_h and bool((acc == 7).all())
    acc = torch.zeros((C, 5), dtype=torch.int64, device=dev)
    ops.parse_shard(op.si, "stats", channels=C, out=(acc, None))
    assert got_stats(acc, None)[0] == want_b


def _small_shards(n_shards, C, kind, recs=5):
    rng = np.random.default_rng(77)
    shards, chips = [], []
    for s in range(n_shards):
        cs = [_chip(rng, 16, 12 + s, C, "uint8" if kind == 1 else "int16", i) for i in range(recs)]
        if kind == 2:
            cs = [(img, lab.astype(np.float32)) for img, lab in cs]
        shards.append(b"".join(_record(img, lab, b"s%dr%d" % (s, i)) for i, (img, lab) in enumerate(cs)))
        chips += cs
    return shards, chips


@pytest.mark.gpu
@pytest.mark.parametrize("kind", (1, 2))
def test_stats_streaming(dev, kind):
    """ShardPipeline at depth 3 over 11 shards, from device memory and from pinned host memory, adds every shard into one
    counter pair; iter_parsed_shards and shard_stats give the same sums."""
    import torch

    from dl_image_segmentation_b200 import ops
    C = 3
    mode = "stats" if kind == 1 else "stats_f32"
    shards, chips = _small_shards(11, C, kind)
    want_b = ref_band_stats([c[0] for c in chips], C)
    want_h = ref_hist([c[1] for c in chips])
    dshards = [torch.from_numpy(np.frombuffer(s, np.uint8).copy()).to(dev) for s in shards]
    host = [torch.from_numpy(np.frombuffer(s, np.uint8).copy()).pin_memory() for s in shards]
    for src in (dshards, host):
        pipe = ops.ShardPipeline(mode, 0, 0, max_records=8, channels=C, device=dev, depth=3, open_ahead=4,
                                 max_shard_bytes=max(len(s) for s in shards))
        statuses = [st[:5].clone() for _, _, st, _ in pipe.run(src)]
        assert len(statuses) == len(shards) and not any(bool(s.any()) for s in statuses)
        bands, bins = got_stats(*pipe.stats_out)
        assert bands == want_b and bins == want_h
    for sized in (True, False):
        kw = dict(img_elems=0, max_records=8) if sized else {}
        res = list(ops.iter_parsed_shards(dshards, mode, channels=C, device=dev, **kw))
        assert res[0][0] is res[-1][0]                       # one counter pair for every shard
        assert got_stats(res[-1][0], res[-1][1]) == (want_b, want_h)
    bands, bins = ops.shard_stats(host, C, kind="bytes" if kind == 1 else "float", max_records=8, device=dev)
    assert bands == [r[:3] for r in want_b] and bins == want_h


@pytest.mark.gpu
def test_shard_stats_all_reduce_single_rank(dev):
    """all_reduce=True under a one-rank process group: the packed counters go through all_reduce and come back equal."""
    import torch.distributed as dist

    from dl_image_segmentation_b200 import ops
    shards, chips = _small_shards(3, 2, 1)
    want = ops.shard_stats(shards, 2, device=dev)
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    try:
        assert ops.shard_stats(shards, 2, device=dev, all_reduce=True) == want
    finally:
        dist.destroy_process_group()
    assert want[0] == [r[:3] for r in ref_band_stats([c[0] for c in chips], 2)]


# ------------------------------------------------------------------------------------------------ full size (GPU)
@pytest.mark.gpu
def test_stats_cfg2_matches_raw_band_stats(dev):
    """16 full-size cfg2 records (256 x 256 x 3 uint8, 10 classes + 2 % nodata 255) built on the device as bench.py
    builds them: mean_std_from_stats over shard_stats is bit-identical with raw + band_stats, and the histogram is the
    labels' bincount."""
    import torch

    from dl_image_segmentation_b200 import ops
    n, S, C, K = 16, 256, 3, 10
    g = torch.Generator(device=dev)
    g.manual_seed(2002)
    imgs = torch.randint(0, 256, (n, S, S, C), dtype=torch.uint8, device=dev, generator=g)
    labs = torch.randint(0, K, (n, S, S), dtype=torch.uint8, device=dev, generator=g)
    labs[torch.rand((n, S, S), device=dev, generator=g) < 0.02] = 255
    items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=1, h=S, w=S, c=C, th=S, tw=S,
                  identifier=b"256:2:1.0:43:0:%d" % i) for i in range(n)]
    buf, _, total = ops.build_records(items, dev)
    shard = buf[:total].clone()
    bands, hist = ops.shard_stats([shard], C, device=dev)
    si = ops.open_shard(shard, dev)
    raw, _, _ = ops.parse_shard(si, "raw", verify_crc=False)
    acc = ops.band_stats(raw[:, :S * S * C].reshape(-1, C), device=dev)
    want = ops.stats_to_python(acc)
    assert bands == want
    for a, b in zip(ops.mean_std_from_stats(bands), ops.mean_std_from_stats(want)):
        assert a.tobytes() == b.tobytes()
    assert hist == [int(v) for v in np.bincount(labs.cpu().numpy().reshape(-1), minlength=257)]


@pytest.mark.gpu
def test_stats_cfg3_exact(dev):
    """8 cfg3 records (512 x 512 x 4 uint16 as packed FloatList) built on the device: exact against the source arrays."""
    import torch

    from dl_image_segmentation_b200 import ops
    n, S, B = 8, 512, 4
    g = torch.Generator(device=dev)
    g.manual_seed(3303)
    imgs = torch.randint(0, 65536, (n, S, S, B), dtype=torch.int32, device=dev, generator=g).to(torch.uint16)
    labs = torch.randint(0, 10, (n, S, S), dtype=torch.uint8, device=dev, generator=g)
    labs[torch.rand((n, S, S), device=dev, generator=g) < 0.02] = 255
    items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=2, h=S, w=S, c=B, th=S, tw=S,
                  identifier=b"448#32#10.0#43#7#%d" % i) for i in range(n)]
    buf, _, total = ops.build_records(items, dev)
    bands, hist = ops.shard_stats([buf[:total].clone()], B, kind="float", device=dev)
    src = imgs.view(torch.int16).cpu().numpy().view(np.uint16).reshape(-1, B).astype(np.int64)
    assert bands == [(src.shape[0], int(src[:, c].sum()), int((src[:, c] * src[:, c]).sum())) for c in range(B)]
    assert hist == [int(v) for v in np.bincount(labs.cpu().numpy().reshape(-1), minlength=257)]


# ------------------------------------------------------------------------------------------------ misuse, dispatch
@pytest.mark.gpu
def test_stats_misuse(dev):
    """Band counts outside 1..64, misaligned counters and non-zero strides are refused; an unknown kind is a ValueError."""
    import torch

    from dl_image_segmentation_b200 import _lib, ops
    from dl_image_segmentation_b200._lib import B2Error
    op = _opened(3, "uint8", dev)
    for C in (0, 65):
        with pytest.raises(B2Error, match="1..64 channels"):
            ops.parse_table(op.si.table, "stats", channels=C)
        with pytest.raises(B2Error, match="1..64 channels"):
            ops.parse_shard(op.si, "stats", channels=C)
    acc = torch.zeros((3, 5), dtype=torch.int64, device=dev)
    hist = torch.zeros((258,), dtype=torch.int64, device=dev)
    status = torch.empty((64,), dtype=torch.int32, device=dev)
    ctx = _lib.get_ctx(dev)
    for field, value in (("img_out", acc.data_ptr() + 4), ("tgt_out", hist.data_ptr() + 4), ("img_stride", 40),
                         ("tgt_stride", 8)):
        for mode in ("stats", "stats_f32"):
            sink = ops._make_sink(mode, True, acc, hist[:257], channels=3)
            setattr(sink, field, value)
            rc = _lib.lib().b2_tfrecord_parse_table(ctx.handle, _lib.ptr(op.si.shard), op.si.nbytes, op.si.table.max_records,
                                                   _lib.ptr(op.si.table.table), ctypes.byref(sink), _lib.ptr(status),
                                                   ctx.stream())
            assert rc != 0 and b"8-byte aligned" in _lib.lib().b2_last_error(), (field, mode)
    torch.cuda.synchronize(dev)
    assert not acc.any() and not hist.any()
    with pytest.raises(ValueError):
        ops.shard_stats([op.si.shard], 3, kind="uint8", device=dev)


@pytest.mark.gpu
def test_stats_dispatch(dev, tmp_path):
    """torch.profiler: each statistics mode launches its own fused_parse_kernel instantiation, through both maps."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from dl_image_segmentation_b200 import ops
    ou, of = _opened(3, "uint8", dev), _opened(3, "uint16", dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        ops.parse_shard(ou.si, "stats", channels=3)
        ops.parse_table(ou.si.table, "stats", channels=3)
        ops.parse_shard(of.si, "stats_f32", channels=3)
        ops.parse_table(of.si.table, "stats_f32", channels=3)
        torch.cuda.synchronize()
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    events = json.loads(trace.read_text())["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel" and "b2::" in e.get("name", "")), key=lambda e: e["ts"])
    got = [e["name"].split("b2::", 1)[1].split("(", 1)[0] for e in kernels]
    assert got == ["fused_parse_kernel<4, false>"] * 2 + ["fused_parse_kernel<5, false>"] * 2, got
