"""The fused parse's normalise / one-hot sink and the standalone b2_normalise_onehot against float64 references.

Covers what the chip-shaped tests elsewhere leave out: every band-count branch of the image loop (C % 4, C % 2, odd),
the shared-memory one-hot up to its limit and the generic one-hot beyond it, the exact-division fallback, record
layouts (payloads starting at every residue mod 16, straddling tiles, longer than a CTA's chunk), per-record statuses,
and records longer than 2048 CRC tiles (16 MiB) in the CRC, parse and build kernels.

The references (tests/_sink_refs.py) are restated instead of taken from oracle/normalise.py, so that the oracle is
checked as well: the test_reference_* functions need no GPU.
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
def _exact_table(mean, std):
    """(C, 256) float32 quotients of every u8 value, from exact rationals."""
    out = np.empty((len(mean), 256), np.float32)
    for c, (m, s) in enumerate(zip(np.asarray(mean, np.float32), np.asarray(std, np.float32))):
        for x in range(256):
            d = _round_f32(Fraction(x) - Fraction(float(m)))            # an exact zero difference is +0
            if s == 0:
                out[c, x] = np.nan if d == 0 else math.copysign(math.inf, float(d)) * math.copysign(1.0, float(s))
            else:
                neg = (math.copysign(1.0, float(d)) < 0) != (float(s) < 0)
                out[c, x] = _round_f32(Fraction(float(d)) / Fraction(float(s)), neg)
    return out


REF_MEAN = np.array([100.0, -3.3e4, 127.5, 0.1, 1e6, 100.0, 3.1e7], np.float32)
REF_STD = np.array([47.0, 0.1, 1e-37, 3e38, 0.0, -5.0, 33.3], np.float32)


def test_reference_normalise_matches_exact_rationals():
    want = _exact_table(REF_MEAN, REF_STD)                        # (C, 256)
    x = np.arange(256, dtype=np.uint8)[:, None]
    got = ref_normalise(x, REF_MEAN, REF_STD).T
    assert not _bits_differ(got, want).any(), np.argwhere(_bits_differ(got, want))[:5]
    with np.errstate(all="ignore"):
        orc = onorm.normalise(x, REF_MEAN, REF_STD).T
    assert not _bits_differ(orc, want).any(), np.argwhere(_bits_differ(orc, want))[:5]
    # the table really reaches the edges it is meant to: overflow, subnormal results, NaN, signed zeros
    assert np.isinf(want[2]).any() and np.isnan(want[4]).sum() == 0 and np.isinf(want[4]).all()
    assert ((want[3] != 0) & (np.abs(want[3]) < np.finfo(np.float32).tiny)).any()
    assert np.signbit(want[5][100]) and want[5][100] == 0        # (100 - 100) / -5 is -0
    assert np.isnan(_exact_table([7.0], [0.0])[0, 7])


def test_reference_one_hot_matches_oracle():
    lab8 = np.arange(256, dtype=np.uint8).reshape(16, 16)
    for K in (1, 10, 33, 255, 256):
        np.testing.assert_array_equal(ref_one_hot(lab8, K), onorm.one_hot(lab8, K))
    labf = np.array([0.0, -0.0, 1.0, 2.5, -0.5, -1.0, np.nan, np.inf, -np.inf, 1e10, 9.0, 10.0, 3.0000002], np.float32)
    want = np.zeros((labf.size, 10), np.float32)
    want[0, 0] = want[1, 0] = want[2, 1] = want[10, 9] = 1.0
    np.testing.assert_array_equal(ref_one_hot(labf, 10), want)
    with np.errstate(invalid="ignore"):
        np.testing.assert_array_equal(onorm.one_hot(labf, 10), want)


# ------------------------------------------------------------------------------------------------ shard fixtures
BANDS = (1, 2, 3, 4, 5, 6, 7, 8, 12, 16, 17, 31, 63, 64)
CLASSES = (1, 2, 3, 4, 5, 10, 19, 20, 21, 24, 31, 32, 33, 40, 64, 255, 256)
STATS = ("ordinary", "inexact_mean", "negative_std", "exact_division")
N_REC = 41
SHAPES = ((1, 1), (1, 7), (3, 5), (61, 61), (64, 64))
BIG = {6: (256, 256), 19: (40, 2000), 30: (256, 256)}    # 40 x 2000 x 1 is ten 8 KiB tiles


def _stats(kind, C):
    rng = np.random.default_rng(500 + C)
    mean = rng.uniform(40, 200, C)
    std = rng.uniform(10, 90, C)
    if kind == "inexact_mean":                       # x - mean rounds in float32 (0.1f, 3.1e7) or lies far away
        mean = np.resize([0.1, 1e6, -3.3e4, 3.1e7, 127.3], C)
    elif kind == "negative_std":
        std[::2] = -std[::2]
    elif kind == "exact_division":                   # quotients that overflow, and 0/0: the fast path cannot match
        std[-1] = 1e-37
        if C > 1:
            std[0] = 0.0
    return mean.astype(np.float32), std.astype(np.float32)


def _chip(rng, h, w, C):
    img = rng.integers(0, 256, (h, w, C), dtype=np.uint8)
    lab = np.where(rng.random((h, w)) < 0.5, rng.integers(0, 40, (h, w)), rng.integers(0, 256, (h, w))).astype(np.uint8)
    if h * w >= 256:                                 # every byte value in every band, every label value
        img.reshape(-1, C)[:256] = (np.arange(256)[:, None] + 31 * np.arange(C)) % 256
        lab.reshape(-1)[:256] = rng.permutation(256)
    return img, lab


@functools.lru_cache(maxsize=None)
def _shard(C):
    """41 u8 records of C bands; identifier lengths 0..40 move the payload starts through every residue mod 16."""
    rng = np.random.default_rng(C)
    recs, chips = [], []
    for i in range(N_REC):
        h, w = BIG.get(i, SHAPES[i % len(SHAPES)])
        img, lab = _chip(rng, h, w, C)
        recs.append(_record(img, lab, bytes(rng.integers(97, 123, i, dtype=np.uint8))))
        chips.append((img, lab))
    return b"".join(recs), chips


class _Opened:
    """A shard on the device, opened once, with its payloads on the device for building expectations."""

    def __init__(self, shard, chips, dev, max_records=64):
        import torch

        from dl_image_segmentation_b200 import ops
        self.si = ops.open_shard(shard, dev, max_records=max_records)
        assert self.si.n == len(chips)
        self.chips = chips
        self.x = [torch.from_numpy(img.reshape(-1).copy()).to(dev) for img, _ in chips]
        self.lab = [torch.from_numpy(lab.reshape(-1).copy()).to(dev) for _, lab in chips]
        self.img_elems = max(img.size for img, _ in chips)
        self.tgt_elems = max(lab.size for _, lab in chips)


@functools.lru_cache(maxsize=None)
def _opened(C, dev):
    return _Opened(*_shard(C), dev)


# ------------------------------------------------------------------------------------------------ device comparisons
def _assert_same_bits(got, want, what):
    import torch
    gn, wn = torch.isnan(got), torch.isnan(want)
    bad = ((got.view(torch.int32) != want.view(torch.int32)) & ~(gn & wn)) | (gn != wn)
    n = int(bad.sum())
    if n:
        i = int(bad.nonzero()[0, 0])
        pytest.fail("%s: %d of %d floats differ; first at %d: got %r, want %r" % (what, n, bad.numel(), i, float(got[i]), float(want[i])))


def _expect_img(xs, mean, std, C):
    """Reference quotients of the payload bytes xs (u8 device tensors): ref_normalise tabulated for the 256 x C
    distinct inputs on the CPU, gathered on the device."""
    import torch
    dev = xs[0].device
    lut = torch.from_numpy(ref_normalise(np.arange(256, dtype=np.uint8)[:, None], mean, std).reshape(-1)).to(dev)
    x = torch.cat(xs).long()
    band = torch.cat([torch.arange(t.numel(), device=dev) % C for t in xs])
    return lut[x * C + band]


def _expect_hot(labs, K):
    import torch
    eye = torch.from_numpy(ref_one_hot(np.arange(256, dtype=np.uint8), K)).to(labs[0].device)
    return eye[torch.cat(labs).long()].reshape(-1)


def _check_rows(op, img_buf, tgt_buf, rows, mean, std, C, K, what):
    import torch
    got_i = torch.cat([img_buf[r, :op.x[r].numel()] for r in rows])
    _assert_same_bits(got_i, _expect_img([op.x[r] for r in rows], mean, std, C), what + " image")
    got_t = torch.cat([tgt_buf[r, :op.lab[r].numel() * K] for r in rows])
    _assert_same_bits(got_t, _expect_hot([op.lab[r] for r in rows], K), what + " one-hot")


def _check_fused(op, mean, std, C, K):
    for name, ib, tb, stat in _parse_both(op, "norm_onehot", mean, std, K):
        assert not stat.any(), (name, np.nonzero(stat)[0], stat[np.nonzero(stat)[0]])
        _check_rows(op, ib, tb, range(op.si.n), mean, std, C, K, name)


# ------------------------------------------------------------------------------------------------ fused parse (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("stats", STATS)
@pytest.mark.parametrize("C", BANDS)
def test_fused_norm_onehot_bands(dev, C, stats):
    """Every branch of the image stride (C % 4 == 0, C % 2 == 0, odd C) and the band cycling behind it, with the
    fast quotient and with the exact-division fallback."""
    mean, std = _stats(stats, C)
    _check_fused(_opened(C, dev), mean, std, C, 10)


@pytest.mark.gpu
@pytest.mark.parametrize("K", CLASSES)
@pytest.mark.parametrize("C", (3, 4))
def test_fused_norm_onehot_classes(dev, C, K):
    """The shared-memory one-hot (K <= 32, including its largest blocks at K = 20..32) and the generic path (K > 32)."""
    mean, std = _stats("ordinary", C)
    _check_fused(_opened(C, dev), mean, std, C, K)


@pytest.mark.gpu
def test_fused_statuses_keep_neighbours_exact(dev):
    """Records the sink must refuse get their status; the records around them are still parsed exactly."""
    C, K = 3, 10
    rng = np.random.default_rng(31)
    recs, chips, want = [], [], []

    def add(rec, chip, status):
        recs.append(rec)
        chips.append(chip)
        want.append(status)

    def good(h, w):
        img, lab = _chip(rng, h, w, C)
        add(_record(img, lab, b"good%d" % len(recs)), (img, lab), 0)

    good(64, 64)
    img16 = rng.integers(0, 65536, (8, 8, C)).astype(np.uint16)               # FloatList record
    add(_record(img16, rng.integers(0, 10, (8, 8)).astype(np.uint8), b"float"), _chip(rng, 8, 8, C), 2)
    good(61, 61)
    img, lab = _chip(rng, 64, 64, C)                                          # payload byte flipped after framing
    bad = bytearray(_record(img, lab, b"crc"))
    bad[len(bad) // 2] ^= 0x20
    add(bytes(bad), (img, lab), 1)
    good(3, 5)
    add(_record(*_chip(rng, 20, 20, 4), b"four bands"), _chip(rng, 20, 20, C), 2)
    good(61, 61)
    img, lab = _chip(rng, 10, 10, C)                                          # image/height says 11
    add(_record(img, lab, b"img_len", dims=(11, 10, C, 10, 10)), (img, lab), 2)
    good(1, 7)
    img, lab = _chip(rng, 10, 10, C)                                          # target/height says 9
    add(_record(img, lab, b"tgt_len", dims=(10, 10, C, 9, 10)), (img, lab), 2)
    good(64, 64)
    img, lab = _chip(rng, 100, 100, C)                                        # longer than the rows below
    add(_record(img, lab, b"too long"), (img, lab), 3)
    good(40, 50)
    op = _Opened(b"".join(recs), chips, dev)
    mean, std = _stats("ordinary", C)
    for name, ib, tb, stat in _parse_both(op, "norm_onehot", mean, std, K, img_elems=64 * 64 * C, tgt_elems=64 * 64):
        assert list(stat) == want, name
        _check_rows(op, ib, tb, [r for r, s in enumerate(want) if s == 0], mean, std, C, K, name)


# ------------------------------------------------------------------------------------------------ standalone K4 (GPU)
def _dev_array(arr, dev, offset):
    """arr on the device, `offset` elements into a fresh (aligned) buffer: offset 1 takes the unaligned load paths."""
    import torch
    tdt = {"uint8": torch.uint8, "uint16": torch.uint16, "int16": torch.int16, "float32": torch.float32}[arr.dtype.name]
    esz = arr.dtype.itemsize
    raw = torch.from_numpy(np.frombuffer(np.ascontiguousarray(arr).tobytes(), np.uint8).copy())
    base = torch.zeros((raw.numel() + esz * offset,), dtype=torch.uint8, device=dev)
    base[esz * offset:].copy_(raw)
    t = base[esz * offset:].view(tdt).view(arr.shape)
    assert t.data_ptr() % 16 == esz * offset
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("C", (1, 3, 4, 5, 16, 17, 64))
@pytest.mark.parametrize("dtype", ("uint8", "uint16", "int16", "float32"))
def test_standalone_normalise(dev, dtype, C):
    from dl_image_segmentation_b200 import ops
    rng = np.random.default_rng(C)
    n = 3001
    if dtype == "float32":
        img = (rng.normal(0, 1000, (n, C)) * rng.choice([1e-3, 1.0, 1e30], (n, C))).astype(np.float32)
        special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 3e38, -3e38, 1e-40, 16777217.0, 0.1], np.float32)
        img.reshape(-1)[:special.size * C] = np.repeat(special, C)
    else:
        info = np.iinfo(dtype)
        img = rng.integers(info.min, info.max + 1, (n, C)).astype(dtype)
        img[:256] = np.arange(256)[:, None] if dtype == "uint8" else info.min
        img[256] = info.max
    mean, std = _stats("ordinary", C)
    mean[0] = 0.1
    if C >= 3:
        std[1], std[2] = 0.0, -5.0
    want = ref_normalise(img, mean, std)
    for offset in (0, 1):
        got, _ = ops.normalise_onehot(_dev_array(img, dev, offset), None, mean, std, 1, device=dev)
        bad = _bits_differ(got.cpu().numpy(), want)
        assert not bad.any(), (offset, int(bad.sum()), np.argwhere(bad)[:3])


@pytest.mark.gpu
@pytest.mark.parametrize("K", (1, 3, 24, 25, 40))
@pytest.mark.parametrize("ldtype", ("uint8", "float32"))
def test_standalone_one_hot(dev, ldtype, K):
    """Both sides of the shared-memory block kernel's limit (K = 24 / 25), u8 and float labels."""
    from dl_image_segmentation_b200 import ops
    rng = np.random.default_rng(K)
    n = 256 * 37 + 13                                  # more blocks than one pass of the grid, ragged last block
    if ldtype == "uint8":
        lab = rng.integers(0, 256, n).astype(np.uint8)
        lab[:256] = np.arange(256)
        lab[256:4000] = rng.integers(0, K + 2, 3744)
    else:
        lab = rng.integers(-3, K + 4, n).astype(np.float32)
        special = np.array([0.0, -0.0, 0.5, 2.5, -0.5, -1.0, np.nan, np.inf, -np.inf, 1e10, K, K + 1, K - 0.5, 255.0,
                            16777216.0, 1.0000001, np.finfo(np.float32).tiny], np.float32)
        lab[:special.size] = special
        lab[1000:1000 + 40 * special.size:40] = special
    want = ref_one_hot(lab, K)
    for offset in (0, 1):
        _, got = ops.normalise_onehot(None, _dev_array(lab, dev, offset), None, None, K, device=dev)
        bad = _bits_differ(got.cpu().numpy(), want)
        assert not bad.any(), (offset, int(bad.sum()), np.argwhere(bad)[:3])


# ------------------------------------------------------------------------------------------------ > 2048 tiles (GPU)
@pytest.mark.gpu
def test_crc32c_past_2048_tiles(dev):
    """A CRC partial that has to move 2048 tiles (16 MiB) or more goes through x^(8n) by squaring, not the table."""
    from dl_image_segmentation_b200 import ops
    lens = [(16 << 20) + 1, (16 << 20) - 7, 40_000_003, 8192 * 2049 + 5]
    rng = np.random.default_rng(16)
    data = rng.integers(0, 256, sum(lens) + 64, dtype=np.uint8)
    offs, p = [], 3
    for ln in lens:
        offs.append(p)
        p += ln + 9                                    # odd starts
    got = ops.crc32c(data, offs, lens, device=dev)
    assert [int(g) for g in got] == [otfr.crc32c(data[o:o + ln]) for o, ln in zip(offs, lens)]


@pytest.mark.gpu
def test_parse_record_past_2048_tiles(dev):
    """One ~17 MiB record (2400 x 2400 x 3) and a small one after it, CRC verified, in every sink mode."""
    import torch

    from dl_image_segmentation_b200 import ops
    C, K, h = 3, 3, 2400
    rng = np.random.default_rng(2400)
    chips = [_chip(rng, h, h, C), _chip(rng, 64, 64, C)]
    chips[0][1][:] %= 5                                # classes 0..2 and out-of-range 3, 4
    recs = [_record(img, lab, b"big%d" % i) for i, (img, lab) in enumerate(chips)]
    shard = b"".join(recs)
    op = _Opened(shard, chips, dev, max_records=4)
    assert int(op.si.lens_host[0]) > 2048 * 8192
    _, _, st = ops.parse_shard(op.si, "none", verify_crc=True)
    assert list(st.cpu().numpy()) == [0, 0]
    ib, tb, st = ops.parse_shard(op.si, "raw", verify_crc=True)
    assert list(st.cpu().numpy()) == [0, 0]
    for r in range(2):
        assert torch.equal(ib[r, :op.x[r].numel()], op.x[r]) and torch.equal(tb[r, :op.lab[r].numel()], op.lab[r])
    del ib, tb
    mean, std = _stats("ordinary", C)
    for name, ib, tb, stat in _parse_both(op, "norm_onehot", mean, std, K):
        assert list(stat) == [0, 0], name
        _check_rows(op, ib, tb, [0, 1], mean, std, C, K, name)
    del ib, tb
    # a flipped byte far past the 2048th tile is caught
    bad = bytearray(shard)
    bad[12 + 17_000_000] ^= 0x01
    si = ops.open_shard(bytes(bad), dev, max_records=4)
    assert list(ops.parse_shard(si, "none", verify_crc=True)[2].cpu().numpy()) == [1, 0]


@pytest.mark.gpu
def test_build_record_past_2048_tiles(dev):
    """A FloatList record of ~19 MiB (1100 x 1100 x 4 uint16) built on the device is byte-identical with the oracle."""
    from dl_image_segmentation_b200 import _tfrecord_image_translation as tr
    from dl_image_segmentation_b200 import ops
    rng = np.random.default_rng(1100)
    pairs = [(rng.integers(0, 65536, (1100, 1100, 4)).astype(np.uint16), rng.integers(0, 256, (1100, 1100)).astype(np.uint8)),
             (rng.integers(0, 65536, (9, 7, 4)).astype(np.uint16), rng.integers(0, 256, (9, 7)).astype(np.uint8))]
    items, want = [], b""
    for i, (img, lab) in enumerate(pairs):
        h, w, c = img.shape
        items.append(tr.convert_to_example(img, lab, h, w, c, h, w, "k%d" % i).build_item(dev))
        want += otfr.frame(oep.convert_to_example(img, lab, h, w, c, h, w, "k%d" % i).SerializeToString())
    assert len(want) > 2048 * 8192
    buf, offs, total = ops.build_records(items, dev)
    assert total == len(want)
    assert bytes(buf[:total].cpu().numpy()) == want
