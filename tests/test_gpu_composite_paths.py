"""-m gpu: every dispatch path of the K3 compositors and of K4 b2_band_stats against exact references.

The host dispatchers pick a template instantiation from T, B, the element type, hw, the chip count and pointer
alignment.  Each table below names the kernel a case must run, `test_dispatch_paths` checks that name under
torch.profiler, and every other test compares the result exactly with a plain reference:
- the masked median with np.ma.median in float64 (oracle.composite.median_composite);
- the mosaic with the oracle's painter's loop, whose day arithmetic is in Python ints;
- the band statistics with Python-int sums (oracle.normalise.band_stats).
"""
import json

import numpy as np
import pytest

from oracle import composite as ocomp
from oracle import normalise as onorm

pytestmark = pytest.mark.gpu

I32_MIN, I32_MAX = -(1 << 31), (1 << 31) - 1


def _torch_dtype(np_dtype):
    import torch
    return torch.from_numpy(np.empty(0, np_dtype)).dtype


def _placed(x, dev, offset):
    """x on the device as a contiguous view that starts `offset` bytes past a 256-byte boundary."""
    import torch
    x = np.ascontiguousarray(x)
    raw = torch.from_numpy(x.reshape(-1).view(np.uint8))
    buf = torch.empty(raw.numel() + 256, dtype=torch.uint8, device=dev)
    assert buf.data_ptr() % 256 == 0
    v = buf[offset:offset + raw.numel()]
    v.copy_(raw)
    return v.view(_torch_dtype(x.dtype)).view(x.shape)


# ------------------------------------------------------------------------------------------------ K3a masked median
MEDIAN_T = [1, 2, 3, 4, 5, 8, 9, 16, 17, 31, 32, 33]
MEDIAN_B = [1, 2, 3, 4, 6, 8, 16]
MEDIAN_HW = (13, 23)          # hw = 299: hw * B / 2 threads never fill the last 256-thread CTA


def _median_path(T, B, nodata, aligned=True):
    """The kernel b2_median_composite_u16 runs: P = T rounded up to a power of two (at least 2), GPP = B / 2 threads
    per pixel when that is 1, 2, 4 or 8 and 0 otherwise, and the generic kernel for T > 32, odd B or misalignment."""
    P = 2
    while P < T:
        P *= 2
    if P > 32 or B % 2 or not aligned:
        return ("median_generic_kernel",)
    gpp = B // 2 if B // 2 in (1, 2, 4, 8) else 0
    return ("median_kernel<%d, %d, %s, %s>" % (P, gpp, str(nodata).lower(), str(T == P).lower()),)


def _median_inputs(seed, T, B, H, W):
    """Half uniform samples, half from {0, 1, 65534, 65535} so that real samples tie with the kernel's sentinels;
    row 0 has every scene valid, row 1 none, row 2 exactly one.  Non-zero validity and nodata bytes vary."""
    rng = np.random.default_rng(seed)
    uni = rng.integers(0, 65536, (T, H, W, B), dtype=np.uint16)
    ext = rng.choice(np.array([0, 1, 65534, 65535], np.uint16), (T, H, W, B))
    stack = np.where(rng.random((T, H, W, B)) < 0.5, uni, ext)
    valid = (rng.random((T, H, W)) < 0.5) * rng.integers(1, 256, (T, H, W))
    valid[:, 0] = 1
    valid[:, 1] = 0
    valid[:, 2] = 0
    valid[rng.integers(0, T, W), 2, np.arange(W)] = 255
    nodata = (rng.random((T, H, W, B)) < 0.2) * rng.integers(1, 256, (T, H, W, B))
    return stack, valid.astype(np.uint8), nodata.astype(np.uint8)


def _check_median(dev, stack, valid, nodata=None, on_device=None):
    from dl_image_segmentation_b200 import ops
    s, nd = on_device or (stack, nodata)
    out, mask = ops.median_composite(s, valid, nd, device=dev)
    ref = ocomp.median_composite(stack, valid, nodata)
    np.testing.assert_array_equal(mask.cpu().numpy(), np.ma.getmaskarray(ref))
    np.testing.assert_array_equal(out.cpu().numpy(), ref.filled(0.0))


@pytest.mark.parametrize("B", MEDIAN_B)
@pytest.mark.parametrize("T", MEDIAN_T)
def test_median_every_path(dev, T, B):
    stack, valid, nodata = _median_inputs(T * 100 + B, T, B, *MEDIAN_HW)
    _check_median(dev, stack, valid)
    _check_median(dev, stack, valid, nodata)


# (stack offset, nodata offset) in bytes: a stack not 16-byte aligned or a nodata mask not 4-byte aligned takes the
# generic kernel; the offsets stay element-aligned, as any uint16 / uint8 view is
MEDIAN_MISALIGNED = [(2, None), (0, 1), (2, 1)]


@pytest.mark.parametrize("s_off,nd_off", MEDIAN_MISALIGNED)
def test_median_misaligned_inputs(dev, s_off, nd_off):
    stack, valid, nodata = _median_inputs(41, 16, 8, *MEDIAN_HW)
    nodata = None if nd_off is None else nodata
    on_device = (_placed(stack, dev, s_off), None if nodata is None else _placed(nodata, dev, nd_off))
    _check_median(dev, stack, valid, nodata, on_device)


# ------------------------------------------------------------------------------------------------ K3b mosaic
# The cloud fractions and max_cf are exact in float32.  max_cf crosses the C ABI as a float32, so a threshold such as
# 0.7 is compared as float32(0.7) < 0.7 by the kernel but as the double 0.7 by the oracle.
FILTER = dict(ref_day=50, min_day=0, max_day=100, max_cf=0.5)
CFS = np.array([0.0, 0.25, 0.375, 0.5, 0.75], np.float32)

# (dtype, B, H, W, kernel without statistics); 37 x 41 = 1517 pixels (hw % 4 == 1), 36 x 41 = 1476 (hw % 4 == 0)
MOSAIC_LAYOUTS = [
    (np.uint8, 1, 37, 41, "mosaic_kernel<0, 0>"),
    (np.uint8, 3, 37, 41, "mosaic_kernel<0, 0>"),
    (np.uint16, 3, 37, 41, "mosaic_kernel<0, 0>"),
    (np.uint16, 1, 37, 41, "mosaic_kernel<2, 0>"),
    (np.uint8, 2, 37, 41, "mosaic_kernel<2, 0>"),
    (np.uint16, 2, 37, 41, "mosaic_kernel<4, 0>"),
    (np.uint8, 4, 37, 41, "mosaic_kernel<4, 0>"),
    (np.float32, 1, 37, 41, "mosaic_kernel<4, 0>"),
    (np.uint16, 4, 37, 41, "mosaic_kernel<8, 0>"),
    (np.float32, 2, 37, 41, "mosaic_kernel<8, 0>"),
    (np.float64, 1, 37, 41, "mosaic_kernel<8, 0>"),
    (np.uint16, 8, 37, 41, "mosaic_kernel<16, 0>"),
    (np.float32, 4, 37, 41, "mosaic_kernel<16, 0>"),
    (np.float64, 2, 37, 41, "mosaic_kernel<16, 0>"),
    (np.uint16, 4, 36, 41, "mosaic_vec8_kernel<0>"),
    (np.float64, 1, 36, 41, "mosaic_vec8_kernel<0>"),
    (np.uint8, 8, 36, 41, "mosaic_vec8_kernel<0>"),
]
# (dtype, B, H, W, kernels with fused statistics)
MOSAIC_STATS_LAYOUTS = [
    (np.uint8, 2, 37, 41, ("mosaic_kernel<2, 1>",)),
    (np.uint8, 4, 37, 41, ("mosaic_kernel<4, 1>",)),
    (np.uint16, 1, 37, 41, ("mosaic_kernel<2, 2>",)),
    (np.uint16, 2, 37, 41, ("mosaic_kernel<4, 2>",)),
    (np.uint16, 4, 37, 41, ("mosaic_kernel<8, 2>",)),
    (np.uint16, 4, 36, 41, ("mosaic_vec8_kernel<2>", "stats_fold_kernel")),
]


def _lid(layout):
    return "%s-B%d-%dx%d" % (np.dtype(layout[0]).name, layout[1], layout[2], layout[3])


def _mosaic_inputs(seed, n, T, H, W, B, dtype, fill="random"):
    """Random bytes (every bit pattern, NaNs included, for float types), ~35 % validity with varied non-zero bytes,
    days with distance ties around FILTER's ref_day; the last chip has no eligible scene when n > 1."""
    rng = np.random.default_rng(seed)
    dtype = np.dtype(dtype)
    shape = (n, T, H, W, B)
    if fill == "saturated":
        stacks = np.full(shape, np.iinfo(dtype).max, dtype)
        valids = np.ones((n, T, H, W), np.uint8)
    else:
        stacks = rng.integers(0, 256, int(np.prod(shape)) * dtype.itemsize, dtype=np.uint8).view(dtype).reshape(shape)
        valids = ((rng.random((n, T, H, W)) < 0.35) * rng.integers(1, 256, (n, T, H, W))).astype(np.uint8)
    days = rng.integers(-20, 120, (n, T)).astype(np.int32)
    days[:, 0], days[:, -1] = 40, 60                          # a tie at distance 10
    cfs = rng.choice(CFS, (n, T))
    if fill == "saturated":
        days[:], cfs[:] = 50, 0.0
    elif n > 1:
        days[-1] = 200
    return stacks, valids, days, cfs


def _oracle_bounds(flt):
    """min_day / max_day for the oracle: None where the header says the bound is disabled."""
    lo, hi = flt.get("min_day"), flt.get("max_day")
    return (None if lo in (None, I32_MIN) else lo), (None if hi in (None, I32_MAX) else hi)


def _check_mosaic(dev, stacks, valids, days, cfs, flt, acc=None, dev_stacks=None, dev_valids=None):
    """Run the mosaic and compare out (bit for bit), mask, src and n_eligible with the oracle per chip.
    -> (out, mask) on the host."""
    from dl_image_segmentation_b200 import ops
    out, mask, src, nel = ops.nearest_date_mosaic(stacks if dev_stacks is None else dev_stacks,
                                                  valids if dev_valids is None else dev_valids, days, cfs,
                                                  device=dev, stats_acc=acc, **flt)
    o, m, s, ne = out.cpu().numpy(), mask.cpu().numpy(), src.cpu().numpy(), nel.cpu().numpy()
    lo, hi = _oracle_bounds(flt)
    for i in range(len(stacks)):
        order = ocomp.scene_order(days[i], cfs[i], flt["ref_day"], lo, hi, flt.get("max_cf"))
        assert ne[i] == len(order), i
        ref = ocomp.nearest_date_mosaic(stacks[i], valids[i], days[i], cfs[i], flt["ref_day"], lo, hi, flt.get("max_cf"))
        if ref is None:
            T, H, W, B = stacks[i].shape
            ref = np.zeros((H, W, B), stacks[i].dtype), np.ones((H, W), bool), np.full((H, W), -1, np.int16)
        r_out, r_mask, r_src = ref
        np.testing.assert_array_equal(np.ascontiguousarray(o[i]).view(np.uint8), np.ascontiguousarray(r_out).view(np.uint8))
        np.testing.assert_array_equal(m[i], r_mask)
        np.testing.assert_array_equal(s[i], r_src)
    return o, m


def _check_stats(acc, want):
    from dl_image_segmentation_b200 import ops
    got = ops.stats_to_python(acc)
    assert got == want
    for a, b in zip(ops.mean_std_from_stats(got), onorm.mean_std_from_stats(want)):
        np.testing.assert_array_equal(a, b)


def _add_stats(a, b):
    return [tuple(x + y for x, y in zip(p, q)) for p, q in zip(a, b)]


@pytest.mark.parametrize("v_off", [0, 1], ids=["valid-aligned", "valid-off1"])
@pytest.mark.parametrize("layout", MOSAIC_LAYOUTS, ids=_lid)
def test_mosaic_every_layout(dev, layout, v_off):
    """List form; validity planes 4-byte aligned, or 1 byte off (the byte-probe branch of the vec8 kernel)."""
    dtype, B, H, W, _ = layout
    stacks, valids, days, cfs = _mosaic_inputs(B * 10 + v_off, 4, 12, H, W, B, dtype)
    dv = [_placed(v, dev, v_off) for v in valids]
    _check_mosaic(dev, list(stacks), list(valids), days, cfs, FILTER, dev_valids=dv)


# (dtype, B, H, W, kernels) for T in {1, 300, 4096}: the O(T^2) ranking in shared memory up to the ABI's limit
MOSAIC_T_LAYOUTS = [(np.uint16, 4, 6, 10, ("mosaic_vec8_kernel<0>",)), (np.uint8, 3, 7, 9, ("mosaic_kernel<0, 0>",)),
                    (np.uint16, 4, 7, 9, ("mosaic_kernel<8, 2>",))]


@pytest.mark.parametrize("T", [1, 300, 4096])
@pytest.mark.parametrize("layout", MOSAIC_T_LAYOUTS, ids=_lid)
def test_mosaic_scene_counts(dev, layout, T):
    import torch
    dtype, B, H, W, kernels = layout
    stacks, valids, days, cfs = _mosaic_inputs(T + B, 3, T, H, W, B, dtype)
    rng = np.random.default_rng(T)
    days[:2] = rng.integers(-3000, 3000, (2, T))             # ties in |day - 17| at every T > 1
    flt = dict(ref_day=17, min_day=-2500, max_day=2500, max_cf=0.5)
    stats = kernels[0] == "mosaic_kernel<8, 2>"
    acc = torch.zeros((B, 4), dtype=torch.int64, device=dev) if stats else None
    o, m = _check_mosaic(dev, list(stacks), list(valids), days, cfs, flt, acc)
    if stats:
        _check_stats(acc, onorm.band_stats(o.reshape(-1, B), (~m).reshape(-1)))


@pytest.mark.parametrize("fill", ["random", "saturated"])
@pytest.mark.parametrize("layout", MOSAIC_STATS_LAYOUTS, ids=_lid)
def test_mosaic_fused_stats_every_layout(dev, layout, fill):
    """Two calls on different chips accumulate into one acc; saturated = every sample at the type's maximum, all valid."""
    import torch
    dtype, B, H, W, _ = layout
    acc = torch.zeros((B, 4), dtype=torch.int64, device=dev)
    want = [(0, 0, 0)] * B
    for call in range(2):
        stacks, valids, days, cfs = _mosaic_inputs(100 * B + call, 4, 9, H, W, B, dtype, fill)
        o, m = _check_mosaic(dev, list(stacks), list(valids), days, cfs, FILTER, acc)
        want = _add_stats(want, onorm.band_stats(o.reshape(-1, B), (~m).reshape(-1)))
    if fill == "saturated":
        mx, n = np.iinfo(dtype).max, 2 * 4 * H * W
        assert want == [(n, n * mx, n * mx * mx)] * B
    _check_stats(acc, want)


def test_mosaic_fused_stats_chips_share_slots(dev):
    """300 chips: the vec8 kernel's 256 statistics slots are shared through chip & 255 before they are folded."""
    import torch
    n, T, H, W, B = 300, 4, 8, 8, 4
    stacks, valids, days, cfs = _mosaic_inputs(300, n, T, H, W, B, np.uint16)
    acc = torch.zeros((B, 4), dtype=torch.int64, device=dev)
    o, m = _check_mosaic(dev, stacks, valids, days, cfs, FILTER, acc)
    _check_stats(acc, onorm.band_stats(o.reshape(-1, B), (~m).reshape(-1)))


def _ctas_per_chip(sm_count, n_chips, hw):
    """b2_nearest_date_mosaic's CTAs per chip: one per 1024 pixels, at most enough to give the machine 8 per SM."""
    per_chip = (hw + 1023) // 1024
    want = (sm_count * 8 + n_chips - 1) // n_chips
    return (want if want > 0 else 1) if per_chip > want else per_chip


def test_mosaic_fused_stats_vec8_grid_stride_rounds(dev):
    """Enough chips that each gets one CTA, and chips of 1061 groups of 4 pixels: every thread makes three rounds of
    the vec8 grid-stride loop (2 groups per thread per round), the last one ragged.  All chips share one scene list,
    so the oracle paints them as one tall chip."""
    import torch

    from dl_image_segmentation_b200._lib import get_ctx, lib
    sms = lib().b2_ctx_sm_count(get_ctx(dev).handle)
    n, T, H, W, B = 8 * sms, 2, 4, 1061, 4
    per_round = 2 * 256 * _ctas_per_chip(sms, n, H * W)
    groups = H * W // 4
    assert groups > 2 * per_round and groups % per_round, (groups, per_round)
    rng = np.random.default_rng(8)
    stacks = rng.integers(0, 65536, (n, T, H, W, B), dtype=np.uint16)
    valids = (rng.random((n, T, H, W)) < 0.5).astype(np.uint8)
    days = np.tile(np.array([45, 52], np.int32), (n, 1))
    cfs = np.zeros((n, T), np.float32)
    acc = torch.zeros((B, 4), dtype=torch.int64, device=dev)
    from dl_image_segmentation_b200 import ops
    out, mask, src, nel = ops.nearest_date_mosaic(stacks, valids, days, cfs, device=dev, stats_acc=acc, **FILTER)
    tall = lambda a: np.swapaxes(a, 0, 1).reshape((T, n * H) + a.shape[3:])   # noqa: E731
    r_out, r_mask, r_src = ocomp.nearest_date_mosaic(tall(stacks), tall(valids), days[0], cfs[0], 50, 0, 100, 0.5)
    assert (nel.cpu().numpy() == 2).all()
    np.testing.assert_array_equal(out.cpu().numpy().reshape(n * H, W, B), r_out)
    np.testing.assert_array_equal(mask.cpu().numpy().reshape(n * H, W), r_mask)
    np.testing.assert_array_equal(src.cpu().numpy().reshape(n * H, W), r_src)
    _check_stats(acc, onorm.band_stats(r_out.reshape(-1, B), (~r_mask).reshape(-1)))


@pytest.mark.parametrize("dtype,B", [(np.uint8, 1), (np.uint16, 3), (np.uint8, 8), (np.float32, 1)])
def test_mosaic_fused_stats_refusals(dev, dtype, B):
    """Layouts without a fused-statistics kernel raise B2Error and leave acc as it was."""
    import torch

    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    stacks, valids, days, cfs = _mosaic_inputs(5, 2, 3, 8, 8, B, dtype)
    acc = torch.arange(B * 4, dtype=torch.int64, device=dev).reshape(B, 4)
    with pytest.raises(B2Error, match="fused statistics"):
        ops.nearest_date_mosaic(stacks, valids, days, cfs, device=dev, stats_acc=acc, **FILTER)
    torch.cuda.synchronize()
    assert torch.equal(acc.cpu(), torch.arange(B * 4, dtype=torch.int64).reshape(B, 4))


# ------------------------------------------------------------------------------------------------ int32 day edges
EDGE_DAYS = [I32_MIN, I32_MIN + 1, I32_MIN + 2, -2, -1, 0, 1, I32_MAX - 2, I32_MAX - 1, I32_MAX]
EDGE_REFS = [I32_MIN, I32_MIN + 1, -1, 0, I32_MAX - 1, I32_MAX]
EDGE_BOUNDS = [(None, None), (I32_MIN, I32_MAX), (I32_MIN + 1, I32_MAX - 1), (0, None), (None, 0), (I32_MAX - 1, None)]
# both kernels' prologues, with and without statistics
EDGE_LAYOUTS = [(8, 8, False), (5, 7, False), (8, 8, True), (5, 7, True)]


@pytest.mark.parametrize("H,W,stats", EDGE_LAYOUTS)
def test_mosaic_int32_day_edges(dev, H, W, stats):
    import torch
    rng = np.random.default_rng(H * W)
    n, T, B = 3, len(EDGE_DAYS), 4
    stacks = rng.integers(0, 65536, (n, T, H, W, B), dtype=np.uint16)
    valids = (rng.random((n, T, H, W)) < 0.3).astype(np.uint8)
    days = np.stack([rng.permutation(np.array(EDGE_DAYS, np.int64)) for _ in range(n)]).astype(np.int32)
    cfs = np.zeros((n, T), np.float32)
    for ref in EDGE_REFS:
        for lo, hi in EDGE_BOUNDS:
            flt = dict(ref_day=ref)
            if lo is not None:
                flt["min_day"] = lo
            if hi is not None:
                flt["max_day"] = hi
            acc = torch.zeros((B, 4), dtype=torch.int64, device=dev) if stats else None
            o, m = _check_mosaic(dev, stacks, valids, days, cfs, flt, acc)
            if stats:
                _check_stats(acc, onorm.band_stats(o.reshape(-1, B), (~m).reshape(-1)))


@pytest.mark.parametrize("H,W,stats", EDGE_LAYOUTS)
def test_mosaic_int32_max_day_and_far_distances(dev, H, W, stats):
    """A scene dated INT32_MAX is eligible when max_day is None or INT32_MAX, and distances of 2^31 - 2, 2^31 - 1 and
    2^32 - 1 rank by value: the nearer scene wins although the farther one has the higher index."""
    import torch

    from dl_image_segmentation_b200 import ops
    B = 4
    stacks = np.random.default_rng(1).integers(0, 65536, (1, 2, H, W, B), dtype=np.uint16)
    valids = np.ones((1, 2, H, W), np.uint8)
    cfs = np.zeros((1, 2), np.float32)
    for days, ref, bounds, want in [([0, I32_MAX], I32_MAX, {}, 1),
                                    ([0, I32_MAX], I32_MAX, dict(max_day=I32_MAX), 1),
                                    ([0, I32_MAX], I32_MAX, dict(min_day=I32_MIN, max_day=I32_MAX), 1),
                                    ([-1, I32_MAX], I32_MIN, {}, 0),
                                    ([-2, -1], I32_MIN, {}, 0),
                                    ([0, I32_MIN], I32_MAX, {}, 0)]:
        acc = torch.zeros((B, 4), dtype=torch.int64, device=dev) if stats else None
        out, mask, src, nel = ops.nearest_date_mosaic(stacks, valids, np.array([days], np.int32), cfs, ref, device=dev,
                                                      stats_acc=acc, **bounds)
        assert int(nel[0]) == 2, (days, ref, bounds)
        assert (src.cpu().numpy() == want).all(), (days, ref, bounds)
        np.testing.assert_array_equal(out.cpu().numpy()[0], stacks[0, want])


@pytest.mark.parametrize("arg", ["ref_day", "min_day", "max_day"])
@pytest.mark.parametrize("value", [1 << 31, I32_MIN - 1, 1 << 40])
def test_mosaic_day_arguments_outside_int32_raise(dev, arg, value):
    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    stacks, valids, days, cfs = _mosaic_inputs(3, 2, 3, 8, 8, 4, np.uint16)
    flt = dict(FILTER, **{arg: value})
    with pytest.raises(B2Error, match=arg):
        ops.nearest_date_mosaic(stacks, valids, days, cfs, device=dev, **flt)


# (dtype, B, byte offset): each stack must be aligned to its pixel load (2, 4, 8 or 16 bytes; 1 for other sizes)
MISALIGNED_STACKS = [(np.uint8, 2, 1), (np.uint16, 2, 2), (np.uint16, 4, 2), (np.uint16, 4, 4), (np.float32, 2, 4),
                     (np.uint16, 8, 8), (np.float64, 2, 8)]


@pytest.mark.parametrize("dtype,B,offset", MISALIGNED_STACKS)
def test_mosaic_refuses_misaligned_stacks(dev, dtype, B, offset):
    """The check is on the host: nothing is launched for a list holding a misaligned view."""
    from dl_image_segmentation_b200 import ops
    from dl_image_segmentation_b200._lib import B2Error
    stacks, valids, days, cfs = _mosaic_inputs(offset, 2, 3, 8, 8, B, dtype)
    st = [_placed(stacks[0], dev, 0), _placed(stacks[1], dev, offset)]
    with pytest.raises(B2Error, match="aligned"):
        ops.nearest_date_mosaic(st, list(valids), days, cfs, device=dev, **FILTER)


@pytest.mark.parametrize("dtype,B,offset", [(np.uint8, 3, 1), (np.uint16, 3, 2), (np.uint16, 4, 16)])
def test_mosaic_accepts_stacks_aligned_to_their_load(dev, dtype, B, offset):
    """Pixels of 3 or 6 bytes are read byte by byte, so any element-aligned stack is accepted."""
    stacks, valids, days, cfs = _mosaic_inputs(offset, 2, 3, 8, 8, B, dtype)
    st = [_placed(s, dev, offset) for s in stacks]
    _check_mosaic(dev, stacks, valids, days, cfs, FILTER, dev_stacks=st)


# ------------------------------------------------------------------------------------------------ K4 b2_band_stats
# (dtype, B, kernel)
BAND_STATS = [(np.uint8, 1, "stats_kernel<unsigned char, 0>"), (np.uint8, 2, "stats_kernel<unsigned char, 2>"),
              (np.uint8, 3, "stats_kernel<unsigned char, 0>"), (np.uint8, 4, "stats_kernel<unsigned char, 4>"),
              (np.uint8, 8, "stats_kernel<unsigned char, 8>"), (np.uint8, 16, "stats_kernel<unsigned char, 0>"),
              (np.uint16, 1, "stats_kernel<unsigned short, 1>"), (np.uint16, 2, "stats_kernel<unsigned short, 2>"),
              (np.uint16, 3, "stats_kernel<unsigned short, 0>"), (np.uint16, 4, "stats_kernel<unsigned short, 4>"),
              (np.uint16, 8, "stats_kernel<unsigned short, 8>"), (np.uint16, 13, "stats_kernel<unsigned short, 0>"),
              (np.uint16, 16, "stats_kernel<unsigned short, 0>")]


@pytest.mark.parametrize("dtype,B", [c[:2] for c in BAND_STATS], ids=lambda v: np.dtype(v).name if isinstance(v, type) else str(v))
def test_band_stats_every_path(dev, dtype, B):
    """n_pixels % 8 in {0, 1, 7} (the fast path's tail), base 16-byte aligned, 8 but not 16, and one element off
    (the 16-byte loads, the per-pixel vector loads and the scalar loop), with and without a valid mask, for uniform,
    saturated and all-zero samples."""
    from dl_image_segmentation_b200 import ops
    rng = np.random.default_rng(B)
    mx, item = np.iinfo(dtype).max, np.dtype(dtype).itemsize
    for n in (4096, 4097, 4103):
        valid = ((rng.random(n) < 0.7) * rng.integers(1, 256, n)).astype(np.uint8)
        for fill in ("uniform", "saturated", "zero"):
            img = {"uniform": lambda: rng.integers(0, mx + 1, (n, B)).astype(dtype),
                   "saturated": lambda: np.full((n, B), mx, dtype), "zero": lambda: np.zeros((n, B), dtype)}[fill]()
            for offset in (0, 8, item):
                d_img = _placed(img, dev, offset)
                for v in (None, valid):
                    got = ops.stats_to_python(ops.band_stats(d_img, v, device=dev))
                    want = onorm.band_stats(img, v)
                    assert got == want, (n, fill, offset, v is None)
                    for a, b in zip(ops.mean_std_from_stats(got), onorm.mean_std_from_stats(want)):
                        np.testing.assert_array_equal(a, b)


# ------------------------------------------------------------------------------------------------ dispatch paths
def _path_cases(dev):
    """(label, run, kernels) for one case of every table above: `run` launches it once, `kernels` are the b2 kernels
    it must launch, in order."""
    import torch

    from dl_image_segmentation_b200 import ops
    cases = []
    for T in MEDIAN_T:
        for B in MEDIAN_B:
            s, v, nd = _median_inputs(T + B, T, B, 3, 5)
            for with_nd in (False, True):
                cases.append(("median T=%d B=%d nodata=%s" % (T, B, with_nd),
                              lambda s=s, v=v, nd=(nd if with_nd else None): ops.median_composite(s, v, nd, device=dev),
                              _median_path(T, B, with_nd)))
    s, v, nd = _median_inputs(1, 16, 8, 3, 5)
    for s_off, nd_off in MEDIAN_MISALIGNED:
        ds = _placed(s, dev, s_off)
        dnd = None if nd_off is None else _placed(nd, dev, nd_off)
        cases.append(("median misaligned %s/%s" % (s_off, nd_off),
                      lambda ds=ds, dnd=dnd: ops.median_composite(ds, v, dnd, device=dev), ("median_generic_kernel",)))

    def mosaic(dtype, B, H, W, T=5, stats=False, n=2, v_off=0):
        st, va, days, cfs = _mosaic_inputs(B, n, T, H, W, B, dtype)
        dv = [_placed(x, dev, v_off) for x in va]
        acc = torch.zeros((B, 4), dtype=torch.int64, device=dev) if stats else None
        return lambda: ops.nearest_date_mosaic(list(st), dv, days, cfs, device=dev, stats_acc=acc, **FILTER)
    for dtype, B, H, W, k in MOSAIC_LAYOUTS:
        for v_off in (0, 1):
            cases.append(("mosaic %s v_off=%d" % (_lid((dtype, B, H, W)), v_off), mosaic(dtype, B, H, W, v_off=v_off), (k,)))
    for dtype, B, H, W, ks in MOSAIC_T_LAYOUTS:
        for T in (1, 300, 4096):
            stats = ks[0] == "mosaic_kernel<8, 2>"
            cases.append(("mosaic %s T=%d" % (_lid((dtype, B, H, W)), T), mosaic(dtype, B, H, W, T=T, stats=stats, n=3), ks))
    for dtype, B, H, W, ks in MOSAIC_STATS_LAYOUTS:
        cases.append(("mosaic stats %s" % _lid((dtype, B, H, W)), mosaic(dtype, B, H, W, stats=True), ks))
    cases.append(("mosaic stats 300 chips", mosaic(np.uint16, 4, 8, 8, T=4, stats=True, n=300),
                  ("mosaic_vec8_kernel<2>", "stats_fold_kernel")))
    for H, W, stats in EDGE_LAYOUTS:
        ks = {(8, False): "mosaic_vec8_kernel<0>", (7, False): "mosaic_kernel<8, 0>", (8, True): "mosaic_vec8_kernel<2>",
              (7, True): "mosaic_kernel<8, 2>"}[(W, stats)]
        cases.append(("mosaic int32 edges %dx%d stats=%s" % (H, W, stats), mosaic(np.uint16, 4, H, W, stats=stats),
                      (ks, "stats_fold_kernel") if ks == "mosaic_vec8_kernel<2>" else (ks,)))
    for dtype, B, k in BAND_STATS:
        img = np.random.default_rng(B).integers(0, 200, (4097, B)).astype(dtype)
        for offset in (0, 8, np.dtype(dtype).itemsize):
            d_img = _placed(img, dev, offset)
            for valid in (None, np.ones(4097, np.uint8)):
                cases.append(("band_stats %s B=%d offset=%d valid=%s" % (np.dtype(dtype).name, B, offset, valid is not None),
                              lambda d_img=d_img, valid=valid: ops.band_stats(d_img, valid, device=dev), (k,)))
    return cases


def test_dispatch_paths(dev, tmp_path):
    """Every case above runs once under torch.profiler; the b2 kernels it launches must be the ones its table names.
    A change to a dispatch rule that moves a case onto another path fails here, even when the result stays right."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    cases = _path_cases(dev)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _, run, _ in cases:
            run()
        torch.cuda.synchronize()
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    events = json.loads(trace.read_text())["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel" and "b2::" in e.get("name", "")), key=lambda e: e["ts"])
    got = [e["name"].split("b2::", 1)[1].split("(", 1)[0] for e in kernels]
    assert got, "torch.profiler recorded no b2 kernel: the dispatch paths cannot be checked on this machine"
    want = [k for _, _, ks in cases for k in ks]
    if got != want:
        at, i = [], 0
        for label, _, ks in cases:
            if got[i:i + len(ks)] != list(ks):
                at.append("%s: want %s, got %s" % (label, list(ks), got[i:i + len(ks)]))
            i += len(ks)
        pytest.fail("%d kernels recorded, %d expected; first mismatches:\n%s" % (len(got), len(want), "\n".join(at[:10])))
