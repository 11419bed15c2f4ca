"""The fused parse's NORM_ONEHOT_F32 sink: packed float32 FloatList array records (the higher-dtype format the GeoTIFF
path writes) straight to normalised float32 images and one-hot float32 labels, against float64 references.

Every case runs through the uniform tile map (parse_shard) and the opened-table map (parse_table, what ShardPipeline
runs) and is compared bit for bit, NaN matching NaN.  Covers uint16 / int16 / arbitrary float32 bands, every branch of
the image stride, inexact means, negative / zero / tiny stds, class counts on both sides of the shared-memory one-hot,
float labels that have no class, payloads starting at every residue mod 16, per-record statuses, the streaming
readers, a record past 2048 CRC tiles and full-size cfg3 records.

The references are restated in tests/_sink_refs.py; the test_reference_* functions need no GPU.
"""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

from _sink_refs import _bits_differ, _parse_both, _record, _round_f32, ref_normalise, ref_one_hot
from oracle import example_proto as oep
from oracle import normalise as onorm
from oracle import tfrecord as otfr


# ------------------------------------------------------------------------------------------------ references (CPU)
def _exact_quotient(x, m, s):
    """(x - m) / s in float32 arithmetic, from exact rationals, for finite float32 x, m and s."""
    xm = Fraction(float(x)) - Fraction(float(m))
    d = _round_f32(xm, neg=(xm == 0 and math.copysign(1.0, float(x)) < 0 and math.copysign(1.0, float(m)) > 0))
    if s == 0:
        return np.float32(np.nan) if d == 0 else np.float32(math.copysign(math.inf, float(d)) * math.copysign(1.0, float(s)))
    neg = (math.copysign(1.0, float(d)) < 0) != (float(s) < 0)
    return _round_f32(Fraction(float(d)) / Fraction(float(s)), neg)


SPECIAL = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 3e38, -3e38, 1e-40, -1e-45, 16777217.0, 0.1, 65535.0, -32768.0,
                    np.finfo(np.float32).tiny, 1.0000001], np.float32)
LABELS = np.array([0.0, -0.0, 1.0, 2.5, -0.5, -1.0, np.nan, np.inf, -np.inf, 1e10, 9.0, 10.0, 255.0, 3.0000002, 31.0,
                   32.0, 33.0, 255.5, 16777216.0, np.finfo(np.float32).tiny], np.float32)


def test_reference_normalise_matches_exact_rationals():
    mean = np.array([100.0, -3.3e4, 127.5, 0.1, 1e6, 100.0, 3.1e7], np.float32)
    std = np.array([47.0, 0.1, 1e-37, 3e38, 0.0, -5.0, 33.3], np.float32)
    xs = np.concatenate([SPECIAL[np.isfinite(SPECIAL)], np.float32([100.0, 7.25, -2.5e-3, 12345.678, 0.0])])
    got = ref_normalise(xs[:, None], mean, std)
    for i, x in enumerate(xs):
        for c in range(mean.size):
            want = _exact_quotient(x, mean[c], std[c])
            assert not _bits_differ(got[i, c], want), (float(x), c, float(got[i, c]), float(want))
    assert np.signbit(got[list(xs).index(100.0), 5]) and got[list(xs).index(100.0), 5] == 0    # (100 - 100) / -5 is -0


def test_reference_one_hot_values():
    want = np.zeros((LABELS.size, 10), np.float32)
    for i, v in enumerate(LABELS):
        if math.isfinite(v) and v >= 0 and v == int(v) and int(v) < 10:
            want[i, int(v)] = 1.0
    np.testing.assert_array_equal(ref_one_hot(LABELS, 10), want)
    assert want[1, 0] == 1.0 and not want[3].any() and not want[6].any()


@pytest.mark.parametrize("dtype", ("uint16", "int16", "float32"))
def test_reference_matches_oracle_float_records(dtype):
    """The oracle's route for a FloatList record: parse_higher_dtype_array_proto, then normalise and one_hot."""
    rng = np.random.default_rng(7)
    C, K, h, w = 3, 10, 5, 7
    mean, std = _stats("zero_std", C)
    imgs, labs, recs = [], [], []
    for i in range(3):
        img, lab = _chip(rng, h, w, C, dtype)
        imgs.append(img)
        labs.append(lab)
        recs.append(oep.convert_to_example(img, lab, h, w, C, h, w, b"r%d" % i).SerializeToString())
    for i, r in enumerate(recs):
        img, tgt, _ = oep.parse_higher_dtype_array_proto(r)
        assert img.dtype == np.float32 and tgt.dtype == np.float32
        with np.errstate(all="ignore"):
            oi, oh = onorm.normalise(img, mean, std), onorm.one_hot(tgt, K)
        assert not _bits_differ(oi, ref_normalise(imgs[i], mean, std)).any()
        np.testing.assert_array_equal(oh, ref_one_hot(labs[i], K))


# ------------------------------------------------------------------------------------------------ shard fixtures
BANDS = (1, 2, 3, 4, 5, 7, 8, 13, 64)
DTYPES = ("uint16", "int16", "float32")
STATS = ("ordinary", "inexact_mean", "negative_std", "zero_std")
CLASSES = (1, 2, 10, 20, 24, 25, 31, 32, 33, 256)
N_REC = 41
SHAPES = ((1, 1), (1, 7), (3, 5), (29, 31), (32, 32))
BIG = {6: (96, 96), 19: (20, 1100), 30: (64, 64)}    # 20 x 1100 x 1 float32 is eleven 8 KiB tiles


def _stats(kind, C):
    rng = np.random.default_rng(700 + C)
    mean = rng.uniform(40, 200, C)
    std = rng.uniform(10, 90, C)
    if kind == "inexact_mean":                       # x - mean rounds in float32
        mean = np.resize([0.1, 1e6, -3.3e4, 3.1e7, 127.3], C)
    elif kind == "negative_std":
        std[::2] = -std[::2]
    elif kind == "zero_std":
        std[-1] = 1e-37
        if C > 1:
            std[0] = 0.0
    return mean.astype(np.float32), std.astype(np.float32)


def _chip(rng, h, w, C, dtype, K=40):
    n = h * w * C
    if dtype == "float32":
        img = (rng.normal(0, 1000, n) * rng.choice([1e-3, 1.0, 1e30], n)).astype(np.float32)
        k = min(n, SPECIAL.size)
        img[:k] = SPECIAL[:k]
        img = img.reshape(h, w, C)
    else:
        info = np.iinfo(dtype)
        img = rng.integers(info.min, info.max + 1, (h, w, C)).astype(dtype)
        img.reshape(-1)[:2] = np.array([info.min, info.max], dtype)[:min(n, 2)]
    lab = np.where(rng.random((h, w)) < 0.7, rng.integers(0, K + 3, (h, w)), 255).astype(np.float32)
    k = min(lab.size, LABELS.size)
    lab.reshape(-1)[:k] = rng.permutation(LABELS)[:k]
    return img, lab


@functools.lru_cache(maxsize=None)
def _shard(C, dtype, K=40):
    """41 FloatList records of C bands; identifier lengths 0..40 move the payload starts through every residue mod 16."""
    rng = np.random.default_rng(1000 * C + len(dtype))
    recs, chips = [], []
    for i in range(N_REC):
        h, w = BIG.get(i, SHAPES[i % len(SHAPES)])
        if C >= 13 and i in BIG:
            h, w = 24, 24
        img, lab = _chip(rng, h, w, C, dtype, K)
        recs.append(_record(img, lab, bytes(rng.integers(97, 123, i, dtype=np.uint8))))
        chips.append((img, lab))
    return b"".join(recs), chips


class _Opened:
    def __init__(self, shard, chips, dev, max_records=64):
        from dl_image_segmentation_b200 import ops
        self.shard = shard
        self.si = ops.open_shard(shard, dev, max_records=max_records)
        assert self.si.n == len(chips)
        self.chips = chips
        self.img_elems = max(img.size for img, _ in chips)
        self.tgt_elems = max(lab.size for _, lab in chips)


@functools.lru_cache(maxsize=None)
def _opened(C, dtype, dev):
    return _Opened(*_shard(C, dtype), dev)


def _check_rows(chips, img_buf, tgt_buf, rows, mean, std, K, what):
    ib, tb = img_buf.cpu().numpy(), tgt_buf.cpu().numpy()
    for r in rows:
        img, lab = chips[r]
        bad = _bits_differ(ib[r, :img.size], ref_normalise(img.reshape(-1, img.shape[-1]), mean, std).reshape(-1))
        assert not bad.any(), (what, "image", r, int(bad.sum()), np.argwhere(bad)[:3].ravel())
        bad = _bits_differ(tb[r, :lab.size * K], ref_one_hot(lab, K).reshape(-1))
        assert not bad.any(), (what, "one-hot", r, int(bad.sum()), np.argwhere(bad)[:3].ravel())


def _check_fused(op, mean, std, K):
    for name, ib, tb, stat in _parse_both(op, "norm_onehot_f32", mean, std, K):
        assert not stat.any(), (name, np.nonzero(stat)[0], stat[np.nonzero(stat)[0]])
        _check_rows(op.chips, ib, tb, range(op.si.n), mean, std, K, name)


# ------------------------------------------------------------------------------------------------ fused parse (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("stats", STATS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", BANDS)
def test_fused_f32_bands(dev, C, dtype, stats):
    """Every branch of the image stride and its band cycle; uint16 / int16 / arbitrary float32 values."""
    mean, std = _stats(stats, C)
    _check_fused(_opened(C, dtype, dev), mean, std, 10)


@pytest.mark.gpu
@pytest.mark.parametrize("K", CLASSES)
def test_fused_f32_classes(dev, K):
    """The shared-memory one-hot (K <= 32, its largest blocks at K = 20..32) and the generic path (K > 32), with float
    labels in and out of range, 255, non-integral, negative, -0.0, NaN and +-inf."""
    C = 4
    mean, std = _stats("ordinary", C)
    _check_fused(_opened(C, "uint16", dev), mean, std, K)


@pytest.mark.gpu
def test_fused_f32_matches_raw_then_normalise_onehot(dev):
    """The same shard parsed raw and then normalised / one-hot by b2_normalise_onehot gives the same bits."""
    import torch

    from dl_image_segmentation_b200 import ops
    C, K = 5, 24
    op = _opened(C, "float32", dev)
    mean, std = _stats("inexact_mean", C)
    n = op.si.n
    rb, rt, rst = ops.parse_table(op.si.table, "raw", 4 * op.img_elems, 4 * op.tgt_elems)
    assert not rst[:n].any()
    for name, ib, tb, stat in _parse_both(op, "norm_onehot_f32", mean, std, K):
        assert not stat.any(), name
        for r, (img, lab) in enumerate(op.chips):
            x = rb[r, :4 * img.size].clone().view(torch.float32).view(img.shape)
            y = rt[r, :4 * lab.size].clone().view(torch.float32).view(lab.shape)
            wi, wt = ops.normalise_onehot(x, y, mean, std, K, device=dev)
            assert not _bits_differ(ib[r, :img.size].cpu().numpy(), wi.reshape(-1).cpu().numpy()).any(), (name, r)
            assert torch.equal(tb[r, :lab.size * K], wt.reshape(-1)), (name, r)


@pytest.mark.gpu
def test_fused_f32_statuses_keep_neighbours_exact(dev):
    """Records the sink must refuse get their status; the records around them are still parsed exactly."""
    C, K = 4, 10
    rng = np.random.default_rng(41)
    recs, chips, want = [], [], []

    def add(rec, chip, status):
        recs.append(rec)
        chips.append(chip)
        want.append(status)

    def good(h, w):
        img, lab = _chip(rng, h, w, C, "uint16")
        add(_record(img, lab, b"good%d" % len(recs)), (img, lab), 0)

    good(32, 32)
    img8 = rng.integers(0, 256, (8, 8, C), dtype=np.uint8)                   # BytesList u8 record
    add(_record(img8, rng.integers(0, 10, (8, 8)).astype(np.uint8), b"bytes"), _chip(rng, 8, 8, C, "uint16"), 2)
    good(29, 31)
    add(_record(*_chip(rng, 20, 20, 3, "uint16"), b"three bands"), _chip(rng, 20, 20, C, "uint16"), 2)
    good(3, 5)
    img, lab = _chip(rng, 10, 10, C, "uint16")                                # image/height says 11
    add(_record(img, lab, b"img_len", dims=(11, 10, C, 10, 10)), (img, lab), 2)
    good(1, 7)
    img, lab = _chip(rng, 10, 10, C, "uint16")                                # target/height says 9
    add(_record(img, lab, b"tgt_len", dims=(10, 10, C, 9, 10)), (img, lab), 2)
    good(32, 32)
    img, lab = _chip(rng, 4, 4, C, "uint16")                                  # unpacked FloatList image
    ex = oep.convert_to_example(img, lab, 4, 4, C, 4, 4, b"unpacked")
    ex.features["image/image_data"] = _UnpackedFloats(img.astype(np.float32).ravel())
    add(otfr.frame(ex.SerializeToString()), (img, lab), 2)
    good(17, 3)
    img, lab = _chip(rng, 32, 32, C, "uint16")                                # payload byte flipped after framing
    bad = bytearray(_record(img, lab, b"crc"))
    bad[len(bad) // 2] ^= 0x20
    add(bytes(bad), (img, lab), 1)
    good(32, 32)
    img, lab = _chip(rng, 40, 40, C, "uint16")                                # longer than the rows below
    add(_record(img, lab, b"too long"), (img, lab), 3)
    good(24, 30)
    op = _Opened(b"".join(recs), chips, dev)
    mean, std = _stats("ordinary", C)
    for name, ib, tb, stat in _parse_both(op, "norm_onehot_f32", mean, std, K, img_elems=32 * 32 * C, tgt_elems=32 * 32):
        assert list(stat) == want, name
        _check_rows(chips, ib, tb, [r for r, s in enumerate(want) if s == 0], mean, std, K, name)


class _UnpackedFloats:
    """A FloatList feature with one float per tag (field 1, wire type 5) instead of one packed run."""

    def __init__(self, values):
        self.values = np.asarray(values, "<f4")

    def serialize(self):
        body = b"".join(b"\x0d" + v.tobytes() for v in self.values)
        return oep._len_field(2, body)                                        # Feature.float_list


@pytest.mark.gpu
def test_fused_f32_record_past_2048_tiles(dev):
    """One ~19 MiB FloatList record (1100 x 1100 x 4 uint16) and a small one after it, CRC verified."""
    C, K = 4, 10
    rng = np.random.default_rng(1100)
    chips = [_chip(rng, 1100, 1100, C, "uint16", K), _chip(rng, 9, 7, C, "uint16", K)]
    shard = b"".join(_record(img, lab, b"big%d" % i) for i, (img, lab) in enumerate(chips))
    op = _Opened(shard, chips, dev, max_records=4)
    assert int(op.si.lens_host[0]) > 2048 * 8192
    mean, std = _stats("inexact_mean", C)
    for name, ib, tb, stat in _parse_both(op, "norm_onehot_f32", mean, std, K):
        assert list(stat) == [0, 0], name
        _check_rows(chips, ib, tb, [0, 1], mean, std, K, name)


# ------------------------------------------------------------------------------------------------ streaming (GPU)
def _small_shards(n_shards, C, K, recs_per_shard=5, h=16, w=12):
    rng = np.random.default_rng(77)
    shards, chips = [], []
    for s in range(n_shards):
        cs = [_chip(rng, h, w, C, "int16", K) for _ in range(recs_per_shard)]
        shards.append(b"".join(_record(img, lab, b"s%dr%d" % (s, i)) for i, (img, lab) in enumerate(cs)))
        chips.append(cs)
    return shards, chips


@pytest.mark.gpu
def test_f32_streaming_readers(dev):
    """ShardPipeline from pinned host memory over more shards than open_ahead, one CapturedPass replay, and
    iter_parsed_shards without sizes."""
    import torch

    from dl_image_segmentation_b200 import ops
    C, K, h, w, R = 3, 20, 16, 12, 5
    mean, std = _stats("negative_std", C)
    shards, chips = _small_shards(11, C, K, R, h, w)
    host = [torch.from_numpy(np.frombuffer(s, np.uint8).copy()).pin_memory() for s in shards]
    pipe = ops.ShardPipeline("norm_onehot_f32", h * w * C, h * w, max_records=8, mean=mean, std=std, num_classes=K,
                             device=dev, open_ahead=4, max_shard_bytes=max(len(s) for s in shards))
    seen = 0
    for k, (ib, tb, st, table) in enumerate(pipe.run(host)):
        assert not st[:R].any() and table.header()[0] == R
        _check_rows(chips[k], ib, tb, range(R), mean, std, K, "pipeline %d" % k)
        seen += 1
    assert seen == len(shards)

    dshards = [torch.from_numpy(np.frombuffer(s, np.uint8).copy()).to(dev) for s in shards[:4]]
    pipe2 = ops.ShardPipeline("norm_onehot_f32", h * w * C, h * w, max_records=8, mean=mean, std=std, num_classes=K,
                              device=dev, depth=4, open_ahead=4)
    cap = ops.CapturedPass(pipe2, dshards, consume=lambda ib, tb, st, t: (ib, tb, st))
    for ib, tb, st in cap.replay():
        ib.zero_()
        tb.zero_()
        st.fill_(-1)
    for k, (ib, tb, st) in enumerate(cap.replay()):
        torch.cuda.synchronize(dev)
        assert not st[:R].any()
        _check_rows(chips[k], ib, tb, range(R), mean, std, K, "captured %d" % k)

    for k, (ib, tb, st, si) in enumerate(ops.iter_parsed_shards(dshards, "norm_onehot_f32", mean=mean, std=std,
                                                                 num_classes=K, device=dev)):
        assert not st.any() and si.n == R
        _check_rows(chips[k], ib, tb, range(R), mean, std, K, "iter %d" % k)


# ------------------------------------------------------------------------------------------------ full size (GPU)
@pytest.mark.gpu
def test_f32_cfg3_full_size(dev):
    """16 cfg3 records (512 x 512 x 4 uint16, labels with 2 % nodata 255) built on the device: the fused mode against
    raw + b2_normalise_onehot for every record, against the CPU reference for two."""
    import torch

    from dl_image_segmentation_b200 import ops
    n, S, B, K = 16, 512, 4, 10
    g = torch.Generator(device=dev)
    g.manual_seed(3303)
    imgs = torch.randint(0, 65536, (n, S, S, B), dtype=torch.int32, device=dev, generator=g).to(torch.uint16)
    labs = torch.randint(0, K, (n, S, S), dtype=torch.uint8, device=dev, generator=g)
    labs[torch.rand((n, S, S), device=dev, generator=g) < 0.02] = 255
    items = [dict(img=imgs[i].reshape(-1), tgt=labs[i].reshape(-1), kind=2, h=S, w=S, c=B, th=S, tw=S,
                  identifier=b"448#32#10.0#43#7#%d" % i) for i in range(n)]
    buf, offs, total = ops.build_records(items, dev)
    st = ops.open_shard_async(buf[:total], dev, max_records=n)
    mean = np.array([3000.5, 2800.25, 2500.0, 4000.1], np.float32)
    std = np.array([1500.0, 1300.3, -1200.0, 2100.7], np.float32)
    ib, tb, status = ops.parse_table(st, "norm_onehot_f32", S * S * B, S * S, mean=mean, std=std, num_classes=K)
    assert st.check("cfg3 shard") == n and not status.any()
    rb, rt, rst = ops.parse_table(st, "raw", S * S * B * 4, S * S * 4)
    assert not rst.any()
    x = rb[:, :S * S * B * 4].contiguous().view(torch.float32).view(n, S, S, B)
    y = rt[:, :S * S * 4].contiguous().view(torch.float32).view(n, S, S)
    wi, wt = ops.normalise_onehot(x, y, mean, std, K, device=dev)
    assert torch.equal(ib.view(n, S, S, B), wi) and torch.equal(tb.view(n, S, S, K), wt)
    chips = [(imgs[i].cpu().numpy(), labs[i].cpu().numpy().astype(np.float32)) for i in (0, n - 1)]
    _check_rows(chips, ib[[0, n - 1]], tb[[0, n - 1]], [0, 1], mean, std, K, "cfg3")
