"""Float64 references and helpers shared by the fused parse sink tests (test_gpu_parse_sinks.py for NORM_ONEHOT,
test_gpu_parse_float_sinks.py for NORM_ONEHOT_F32).

The references are restated here instead of taken from oracle/normalise.py, so that the oracle is checked as well.
"""
import math
from fractions import Fraction

import numpy as np

from oracle import example_proto as oep
from oracle import tfrecord as otfr


def ref_normalise(x, mean, std):
    """(float32(x) - mean) / std per band (last axis), rounded to float32 after the subtraction and after the division.

    Computed in float64: a float64 result of one +, - or / of float32 operands, rounded to float32, is the correctly
    rounded float32 result (float64 has at least 2*24 + 2 bits), so this is IEEE float32 arithmetic.  std = 0 gives
    +-inf or NaN."""
    x = np.asarray(x)
    mean = np.asarray(mean, np.float32).astype(np.float64)
    std = np.asarray(std, np.float32).astype(np.float64)
    with np.errstate(all="ignore"):
        d = (x.astype(np.float32).astype(np.float64) - mean).astype(np.float32)
        return (d.astype(np.float64) / std).astype(np.float32)


def ref_one_hot(label, K):
    """Row k is 1.0 iff the label's value equals k: NaN, +-inf, negative, non-integral and >= K labels give a zero row,
    -0.0 is class 0."""
    lab = np.asarray(label)
    if lab.dtype.kind == "f":
        return (lab.astype(np.float64)[..., None] == np.arange(K, dtype=np.float64)).astype(np.float32)
    return (lab.astype(np.int64)[..., None] == np.arange(K, dtype=np.int64)).astype(np.float32)


def _round_f32(q, neg=False):
    """Exact rational -> float32, round to nearest even; subnormals, underflow to a signed zero, overflow to inf."""
    if q == 0:
        return np.float32(-0.0 if neg else 0.0)
    s = -1.0 if q < 0 else 1.0
    a = abs(q)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    while Fraction(2) ** e > a:
        e -= 1
    while Fraction(2) ** (e + 1) <= a:
        e += 1
    u = max(e - 23, -149)                       # exponent of one unit in the last place (subnormals: 2^-149)
    m = round(a / Fraction(2) ** u)             # Fraction.__round__: ties to even
    v = m * Fraction(2) ** u
    if v >= Fraction(2) ** 128:
        return np.float32(s * math.inf)
    return np.float32(math.copysign(float(v), s))


def _bits_differ(got, want):
    """Positions where two float32 arrays differ bit for bit; NaN matches NaN whatever the payload."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    gn, wn = np.isnan(got), np.isnan(want)
    return (got.view(np.uint32) != want.view(np.uint32)) & ~(gn & wn) | (gn != wn)


def _record(img, lab, ident, dims=None):
    h, w, c = img.shape
    th, tw = lab.shape
    h, w, c, th, tw = dims or (h, w, c, th, tw)
    return otfr.frame(oep.convert_to_example(img, lab, h, w, c, th, tw, ident).SerializeToString())


def _parse_both(op, mode, mean, std, K, img_elems=None, tgt_elems=None):
    """Yield (name, img_buf, tgt_buf, status) from the uniform tile map (parse_shard) and the opened-table map
    (parse_table, what ShardPipeline runs), both in sink mode `mode`."""
    import torch

    from dl_image_segmentation_b200 import ops
    n = op.si.n
    il = op.img_elems if img_elems is None else img_elems
    tl = op.tgt_elems if tgt_elems is None else tgt_elems
    dev = op.si.shard.device
    out = None
    if img_elems is not None:
        out = (torch.empty((n, il), dtype=torch.float32, device=dev), torch.empty((n, tl * K), dtype=torch.float32, device=dev))
    ib, tb, st = ops.parse_shard(op.si, mode, mean=mean, std=std, num_classes=K, out=out)
    yield "parse_shard", ib, tb, st[:n].cpu().numpy()
    del ib, tb
    # parse_table writes only the rows of the table's records: rows for those are enough
    out = (torch.empty((n, il), dtype=torch.float32, device=dev), torch.empty((n, tl * K), dtype=torch.float32, device=dev))
    ib, tb, st = ops.parse_table(op.si.table, mode, il, tl, mean=mean, std=std, num_classes=K, out=out)
    stat = st[:n].cpu().numpy()
    assert op.si.table.header()[4] == int((stat != 0).sum())
    yield "parse_table", ib, tb, stat
