"""Device operators: thin, typed Python wrappers over the C ABI (include/b2chips.h).

Everything here takes and returns CUDA tensors (torch is the allocator / stream provider only) and
enqueues on torch's current stream.  No function in this module computes on the CPU.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from ._lib import B2Error, check, get_ctx, lib, ptr

_NP2B2 = {np.dtype("uint8"): _lib.B2_U8, np.dtype("uint16"): _lib.B2_U16, np.dtype("int16"): _lib.B2_I16,
          np.dtype("uint32"): _lib.B2_U32, np.dtype("int32"): _lib.B2_I32, np.dtype("float32"): _lib.B2_F32,
          np.dtype("float64"): _lib.B2_F64, np.dtype("int8"): _lib.B2_I8}
_T2NP = {torch.uint8: "uint8", torch.int8: "int8", torch.int16: "int16", torch.int32: "int32",
         torch.float32: "float32", torch.float64: "float64"}
for _n in ("uint16", "uint32"):
    if hasattr(torch, _n):
        _T2NP[getattr(torch, _n)] = _n


def bind_host_to_gpu(device_index):
    """Pin this process to the CPU cores (and so, by first touch, the NUMA node) closest to a GPU.  On a multi-GPU box
    the pinned staging buffers of the streaming paths then sit next to the PCIe root the GPU hangs off, so N ranks
    uploading at once do not funnel through one socket's memory controllers.  Best effort: returns the CPU set or None."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device_index))
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, mask in enumerate(words) for b in range(64) if (int(mask) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


class DataLossError(B2Error):
    """A TFRecord frame or data CRC did not verify (TensorFlow raises tf.errors.DataLossError)."""


def b2_dtype(t) -> int:
    if isinstance(t, torch.Tensor):
        return _NP2B2[np.dtype(_T2NP[t.dtype])]
    return _NP2B2[np.dtype(t.dtype)]


def to_device(x, device=None, dtype=None):
    """numpy array / bytes / torch tensor -> contiguous CUDA tensor (no arithmetic, just a copy)."""
    ctx = get_ctx(device)
    if isinstance(x, (bytes, bytearray, memoryview)):
        x = np.frombuffer(x, dtype=np.uint8)
    if isinstance(x, np.ndarray):
        if dtype is not None:
            x = x.astype(dtype, copy=False)
        if not x.flags.writeable:
            x = x.copy()
        x = torch.from_numpy(np.ascontiguousarray(x))
    if not isinstance(x, torch.Tensor):
        raise TypeError("expected bytes, numpy array or torch tensor, got %r" % type(x))
    return x.to(ctx.device, non_blocking=True).contiguous()


# --------------------------------------------------------------------------------------------- K3
def median_composite(stack, valid, nodata=None, device=None):
    """(T,H,W,B) uint16 + (T,H,W[,1]) uint8 -> ((H,W,B) float64, (H,W,B) bool mask).  b2_median_composite_u16."""
    ctx = get_ctx(device)
    stack = to_device(stack, ctx.device)
    valid = to_device(valid, ctx.device)
    if b2_dtype(stack) != _lib.B2_U16:
        raise B2Error("median_composite: stack must be uint16 (got %s)" % stack.dtype)
    if valid.dim() == 4:
        if valid.shape[-1] != 1:
            raise B2Error("median_composite: valid must be (T,H,W) or (T,H,W,1)")
        valid = valid[..., 0].contiguous()
    if valid.dtype == torch.bool:
        valid = valid.to(torch.uint8)
    T, H, W, B = stack.shape
    if tuple(valid.shape) != (T, H, W) or valid.dtype != torch.uint8:
        raise B2Error("median_composite: valid must be uint8 of shape (T,H,W)")
    nd = None
    if nodata is not None:
        nd = to_device(nodata, ctx.device)
        if nd.dtype == torch.bool:
            nd = nd.to(torch.uint8)
        if tuple(nd.shape) != (T, H, W, B) or nd.dtype != torch.uint8:
            raise B2Error("median_composite: nodata mask must be uint8/bool of shape (T,H,W,B)")
    out = torch.empty((H, W, B), dtype=torch.float64, device=ctx.device)
    mask = torch.empty((H, W, B), dtype=torch.uint8, device=ctx.device)
    check(lib().b2_median_composite_u16(ctx.handle, ptr(stack), ptr(valid), ptr(nd), T, H, W, B, ptr(out), ptr(mask),
                                        ctx.stream()))
    return out, mask.view(torch.bool)


_I32_MIN, _I32_MAX = -(1 << 31), (1 << 31) - 1


def nearest_date_mosaic(stacks, valids, scene_day, scene_cf, ref_day, min_day=None, max_day=None, max_cf=None,
                        device=None, want_src=True, ptr_tables=None, stats_acc=None):
    """Batched nearest-to-reference-date mosaic.  b2_nearest_date_mosaic.

    stacks: (N,T,H,W,B) tensor or list of N (T,H,W,B) tensors; valids: (N,T,H,W) / list of (T,H,W) uint8;
    scene_day (N,T) int32; scene_cf (N,T) float32.  Returns out (N,H,W,B), mask (N,H,W) bool,
    src (N,H,W) int16 or None, n_eligible (N,) int32 — all on the device.  stats_acc: optional (B,4) int64
    CUDA tensor; the band statistics of the valid output pixels are accumulated into it in the same pass.
    Days are int32: a day argument outside that range raises B2Error instead of wrapping to another day.  Each stack
    must be aligned to its pixel's load width (the pixel size when that is 2, 4, 8 or 16 bytes); with ptr_tables the
    tables' pointers are the caller's to align.
    """
    for name, d in (("ref_day", ref_day), ("min_day", min_day), ("max_day", max_day)):
        if d is not None and not _I32_MIN <= int(d) <= _I32_MAX:
            raise B2Error("nearest_date_mosaic: %s = %d is outside int32" % (name, int(d)))
    ctx = get_ctx(device)
    if isinstance(stacks, (list, tuple)):
        st = [to_device(s, ctx.device) for s in stacks]
        va = [to_device(v, ctx.device) for v in valids]
    else:
        s_all = to_device(stacks, ctx.device)
        v_all = to_device(valids, ctx.device)
        st = [s_all[i] for i in range(s_all.shape[0])]
        va = [v_all[i] for i in range(v_all.shape[0])]
    n = len(st)
    T, H, W, B = st[0].shape
    eb = st[0].element_size()
    load = B * eb if B * eb in (2, 4, 8, 16) else 1          # the kernels read a whole pixel of these sizes at once
    for s, v in zip(st, va):
        if tuple(s.shape) != (T, H, W, B) or s.dtype != st[0].dtype or not s.is_contiguous():
            raise B2Error("nearest_date_mosaic: all stacks must be contiguous with one shape and dtype")
        if tuple(v.shape) != (T, H, W) or v.dtype != torch.uint8 or not v.is_contiguous():
            raise B2Error("nearest_date_mosaic: valids must be contiguous uint8 (T,H,W)")
        if ptr_tables is None and s.data_ptr() % load:
            raise B2Error("nearest_date_mosaic: a stack must be aligned to its %d-byte pixels (address %#x)" % (load, s.data_ptr()))
    day = to_device(np.ascontiguousarray(scene_day, dtype=np.int32) if not isinstance(scene_day, torch.Tensor) else scene_day, ctx.device)
    cf = to_device(np.ascontiguousarray(scene_cf, dtype=np.float32) if not isinstance(scene_cf, torch.Tensor) else scene_cf, ctx.device)
    if tuple(day.shape) != (n, T) or tuple(cf.shape) != (n, T) or day.dtype != torch.int32 or cf.dtype != torch.float32:
        raise B2Error("nearest_date_mosaic: scene_day / scene_cf must be (N,T) int32 / float32")
    if ptr_tables is None:
        sp = torch.tensor([s.data_ptr() for s in st], dtype=torch.int64).to(ctx.device)
        vp = torch.tensor([v.data_ptr() for v in va], dtype=torch.int64).to(ctx.device)
    else:
        sp, vp = ptr_tables
    out = torch.empty((n, H, W, B), dtype=st[0].dtype, device=ctx.device)
    mask = torch.empty((n, H, W), dtype=torch.uint8, device=ctx.device)
    src = torch.empty((n, H, W), dtype=torch.int16, device=ctx.device) if want_src else None
    nel = torch.empty((n,), dtype=torch.int32, device=ctx.device)
    check(lib().b2_nearest_date_mosaic(
        ctx.handle, ptr(sp), ptr(vp), ptr(day), ptr(cf), int(ref_day),
        _I32_MIN if min_day is None else int(min_day), _I32_MAX if max_day is None else int(max_day),
        float("nan") if max_cf is None else float(max_cf), n, T, H, W, B, eb, ptr(out), ptr(mask), ptr(src), ptr(nel),
        ptr(stats_acc), ctx.stream()))
    return out, mask.view(torch.bool), src, nel


# --------------------------------------------------------------------------------------------- K4
def _band_constants(mean, std, device, who, C=None):
    """mean / std as float32 device tensors with one entry per band: C of them, or as many as mean has."""
    mean, std = (to_device(np.asarray(v, dtype=np.float32) if not isinstance(v, torch.Tensor) else v, device) for v in (mean, std))
    C = int(mean.numel()) if C is None else C
    if mean.numel() != C or std.numel() != C:
        raise B2Error("%s: mean/std must have one entry per band" % who)
    return mean, std


def normalise_onehot(img, label, mean, std, num_classes, device=None):
    """(N,H,W,C) u8/u16/i16/f32 + (N,H,W) u8/f32 -> ((N,H,W,C) f32, (N,H,W,K) f32).  b2_normalise_onehot."""
    ctx = get_ctx(device)
    img_out = hot = None
    stream = ctx.stream()
    n_pix = None
    if img is not None:
        img = to_device(img, ctx.device)
        C = img.shape[-1]
        mean_d, std_d = _band_constants(mean, std, ctx.device, "normalise_onehot", C)
        img_out = torch.empty(img.shape, dtype=torch.float32, device=ctx.device)
        n_pix = img.numel() // C
        check(lib().b2_normalise_onehot(ctx.handle, ptr(img), b2_dtype(img), None, 0, ptr(mean_d), ptr(std_d), n_pix, C, 1,
                                        ptr(img_out), None, stream))
    if label is not None:
        label = to_device(label, ctx.device)
        if label.dim() >= 3 and label.shape[-1] == 1 and img is not None and label.dim() == img.dim():
            label = label[..., 0].contiguous()
        hot = torch.empty(tuple(label.shape) + (int(num_classes),), dtype=torch.float32, device=ctx.device)
        check(lib().b2_normalise_onehot(ctx.handle, None, 0, ptr(label), b2_dtype(label), None, None, label.numel(), 1,
                                        int(num_classes), None, ptr(hot), stream))
    return img_out, hot


def band_stats(img, valid=None, acc=None, device=None):
    """Accumulate exact integer band statistics into acc (B,4) [int64 storage of uint64 counters]."""
    ctx = get_ctx(device)
    img = to_device(img, ctx.device)
    B = img.shape[-1]
    if acc is None:
        acc = torch.zeros((B, 4), dtype=torch.int64, device=ctx.device)
    v = None
    if valid is not None:
        v = to_device(valid, ctx.device)
        if v.dtype == torch.bool:
            v = v.to(torch.uint8)
    check(lib().b2_band_stats(ctx.handle, ptr(img), b2_dtype(img), ptr(v), img.numel() // B, B, ptr(acc), ctx.stream()))
    return acc


def stats_to_python(acc):
    """(B,4) device counters -> list of (n, sum, sumsq) exact Python ints."""
    a = acc.cpu().numpy().view(np.uint64)
    return [(int(r[0]), int(r[1]), int(r[2]) + 65536 * int(r[3])) for r in a]


def mean_std_from_stats(stats):
    """Exact integer stats -> float32 mean/std (population), each one correctly-rounded float64 division."""
    mean, std = [], []
    for n, s, ss in stats:
        if n == 0:
            mean.append(0.0)
            std.append(1.0)
        else:
            mean.append(s / n)
            std.append(math.sqrt((ss * n - s * s) / (n * n)))
    return np.asarray(mean, dtype=np.float64).astype(np.float32), np.asarray(std, dtype=np.float64).astype(np.float32)


# --------------------------------------------------------------------------------------------- K2
def crc32c(data, offsets, lens, device=None):
    """CRC-32C of byte ranges of a device buffer -> uint32 numpy array (host)."""
    ctx = get_ctx(device)
    data = to_device(data, ctx.device)
    offs = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lens, dtype=np.uint64)
    n = len(offs)
    out = torch.empty((max(n, 1),), dtype=torch.int32, device=ctx.device)
    od = to_device(offs.view(np.int64), ctx.device)
    ld = to_device(ln.view(np.int64), ctx.device)
    check(lib().b2_crc32c(ctx.handle, ptr(data), ptr(od), ptr(ld), n, int(ln.max()) if n else 0, ptr(out), ctx.stream()))
    return out[:n].cpu().numpy().view(np.uint32)


class ShardIndex:
    """A shard resident on the device plus its frame table and per-record feature locations (host copies included)."""

    def __init__(self, shard, nbytes, n, rec_off, rec_len, index_dev, index, lens_host, table=None):
        self.shard, self.nbytes, self.n = shard, nbytes, n
        self.rec_off, self.rec_len, self.index_dev, self.index = rec_off, rec_len, index_dev, index
        self.max_len = int(lens_host.max()) if n else 0
        self.lens_host = lens_host
        self.table = table

    def identifiers(self, shard_host=None):
        """identifier bytes of every record (small D2H gathers)."""
        out = []
        for r in self.index:
            o, l = int(r["id_off"]), int(r["id_len"])
            out.append(bytes(self.shard[o:o + l].cpu().numpy()) if shard_host is None else bytes(shard_host[o:o + l]))
        return out


_layout_cache = {}


def table_layout(nbytes, max_records):
    """(offsets[8]) of a shard table: hdr, rec_off, rec_len, index, tile_start, tile2rec, cap_tiles, total bytes."""
    key = (int(nbytes), int(max_records))
    lay = _layout_cache.get(key)
    if lay is None:
        arr = (ctypes.c_uint64 * 8)()
        check(lib().b2_tfrecord_table_layout(key[0], key[1], arr))
        lay = _layout_cache[key] = tuple(int(x) for x in arr)
        if len(_layout_cache) > 4096:
            _layout_cache.clear()
    return lay


class ShardTable:
    """Device-resident description of one opened shard (b2_tfrecord_open).  Nothing here synchronises until
    header() / fetch() is called, so open -> parse chains can be enqueued shard after shard."""

    def __init__(self, shard, nbytes, max_records, table=None):
        self.shard, self.nbytes, self.max_records = shard, int(nbytes), int(max_records)
        self.layout = table_layout(self.nbytes, self.max_records)
        need = self.layout[7]
        if table is None or table.numel() < need:
            table = torch.empty((need,), dtype=torch.uint8, device=shard.device)
        self.table = table
        self._hdr = None

    def _view(self, k, nbytes, dtype):
        o = self.layout[k]
        return self.table[o:o + nbytes].view(dtype)

    @property
    def hdr_dev(self):
        return self._view(0, 64, torch.int64)

    @property
    def rec_off(self):
        return self._view(1, 8 * self.max_records, torch.int64)

    @property
    def rec_len(self):
        return self._view(2, 8 * self.max_records, torch.int64)

    @property
    def index_dev(self):
        return self._view(3, ctypes.sizeof(_lib.ExampleIndex) * self.max_records, torch.uint8)

    def header(self):
        """(records, scan status, tiles, longest record, records with parse status != 0) — one small D2H read."""
        h = self.hdr_dev.cpu().numpy()
        return int(h[0]), int(h[1]), int(h[2]), int(h[3]), int(h[4])

    def check(self, what="shard"):
        """Raise what TensorFlow raises: DataLossError for a corrupt frame / data CRC, B2Error for a full table."""
        n, st, _, _, bad = self.header()
        if st == 2:
            raise B2Error("%s holds more than max_records=%d records" % (what, self.max_records))
        if st != 0:
            raise DataLossError("corrupted record #%d in %s (bad frame or length CRC)" % (n, what))
        _check_bad_records(bad, what)
        return n


def _check_bad_records(bad, what):
    if bad:
        raise DataLossError("%d record(s) of %s failed the data CRC or the feature template" % (bad, what))


def open_shard_async(data, device=None, max_records=4096, nbytes=None, table=None):
    """Upload (if needed) and enqueue frame scan + feature index on the current stream.  No host synchronisation."""
    ctx = get_ctx(device)
    shard = to_device(data, ctx.device)
    if shard.dtype != torch.uint8 or shard.dim() != 1:
        raise B2Error("open_shard: shard must be a flat uint8 buffer")
    nbytes = int(shard.numel()) if nbytes is None else int(nbytes)
    st = ShardTable(shard, nbytes, max_records, table)
    check(lib().b2_tfrecord_open(ctx.handle, ptr(shard), nbytes, st.max_records, ptr(st.table), ctx.stream()))
    return st


def open_shard(data, device=None, with_index=True, nbytes=None, max_records=4096):
    """Upload (if needed), walk the frames and locate the features; ONE small D2H read-back (the table)."""
    ctx = get_ctx(device)
    cap = int(max_records)
    while True:
        st = open_shard_async(data, ctx.device, cap, nbytes)
        data = st.shard
        lay = st.layout
        host = st.table[:lay[4]].cpu().numpy()          # hdr + rec_off + rec_len + index in one copy
        n, status = int(host[:8].view(np.int64)[0]), int(host[8:16].view(np.int64)[0])
        if status == 2:
            cap *= 16
            continue
        if status != 0:
            raise DataLossError("corrupted record #%d (bad frame or length CRC)" % n)
        break
    lens_host = host[lay[2]:lay[2] + 8 * n].view(np.uint64).copy()
    esz = ctypes.sizeof(_lib.ExampleIndex)
    index = host[lay[3]:lay[3] + esz * n].view(np.dtype(_lib.EXAMPLE_INDEX_DTYPE)).copy() if with_index else None
    return ShardIndex(st.shard, st.nbytes, n, st.rec_off, st.rec_len, st.index_dev if with_index else None, index,
                      lens_host, table=st)


def _align16(x):
    return (int(x) + 15) & ~15


# sink mode -> (b2_parse_sink.mode, payload bytes per element of the normalise / one-hot modes, 0 for the others)
_SINK_MODES = {"none": (_lib.SINK_NONE, 0), "raw": (_lib.SINK_RAW, 0), "norm_onehot": (_lib.SINK_NORM_ONEHOT, 1),
               "norm_onehot_f32": (_lib.SINK_NORM_ONEHOT_F32, 4), "stats": (_lib.SINK_STATS, 0),
               "stats_f32": (_lib.SINK_STATS_F32, 0)}
_STATS_MODES = ("stats", "stats_f32")


def _sink_mode(mode):
    if mode not in _SINK_MODES:
        raise ValueError(mode)
    return _SINK_MODES[mode]


def _float_rows(img_elems, tgt_elems, num_classes):
    """Row lengths (floats) of the normalised image and one-hot buffers for payloads of img_elems / tgt_elems elements:
    the sink needs 16-byte strides, so both are padded to 16 elements unless the rows already are whole 16-byte units."""
    il, tl, K = int(img_elems), int(tgt_elems), int(num_classes)
    if (il * 4) % 16 or (tl * K * 4) % 16:
        il, tl = _align16(il), _align16(tl)
    return il, tl * K


def _stats_out(out, channels, device):
    """The (acc (C,5) int64, hist (257,) int64) counters of the statistics modes: zeroed new ones, or the caller's (either
    may be None: the kernel then skips it)."""
    if out is not None:
        acc, hist = out
        if acc is not None and (acc.dtype != torch.int64 or tuple(acc.shape) != (channels, 5) or not acc.is_contiguous()):
            raise B2Error("statistics counters: acc must be a contiguous (%d, 5) int64 tensor" % channels)
        if hist is not None and (hist.dtype != torch.int64 or tuple(hist.shape) != (257,) or not hist.is_contiguous()):
            raise B2Error("statistics counters: hist must be a contiguous (257,) int64 tensor")
        return acc, hist
    return (torch.zeros((channels, 5), dtype=torch.int64, device=device),
            torch.zeros((257,), dtype=torch.int64, device=device))


def parse_shard(si: ShardIndex, mode, verify_crc=True, mean=None, std=None, num_classes=None, first=0, count=None,
                out=None, channels=None):
    """Run the fused parse kernel over records [first, first+count).  Returns (img_buf, tgt_buf, status_dev).

    mode 'raw': img_buf (count, img_stride) uint8 holding each record's payload bytes as stored;
    mode 'norm_onehot': uint8 BytesList records -> img_buf (count, img_len) float32, tgt_buf (count, tgt_len*K) float32;
    mode 'norm_onehot_f32': packed float32 FloatList records (the higher-dtype array format) -> the same outputs, with
    img_len / tgt_len counted in float elements (the index's byte lengths / 4);
    mode 'stats' (records as 'norm_onehot') / 'stats_f32' (records as 'norm_onehot_f32'): img_buf = acc (channels, 5)
    int64 per-band { n, sum x, sum x^2 lo, sum x^2 hi, excluded }, tgt_buf = hist (257,) int64 label bins (b2chips.h
    B2_SINK_STATS); both accumulate into out=(acc, hist) when it is given.  Defined only if every status is 0;
    mode 'none': CRC verification only.
    """
    ctx = get_ctx(si.shard.device)
    count = si.n - first if count is None else count
    if count <= 0:
        return None, None, None
    _, esz = _sink_mode(mode)
    idx = si.index[first:first + count] if si.index is not None else None
    img_buf = tgt_buf = None
    if mode in _STATS_MODES:
        img_buf, tgt_buf = _stats_out(out, channels, ctx.device)
    elif mode == "raw":
        istr, tstr = _align16(max(1, idx["img_len"].max())), _align16(max(1, idx["tgt_len"].max()))
        img_buf, tgt_buf = out if out is not None else (
            torch.empty((count, istr), dtype=torch.uint8, device=ctx.device),
            torch.empty((count, tstr), dtype=torch.uint8, device=ctx.device))
    elif esz:
        # the band count is the sink's, as in parse_table: a record with another band count gets status 2
        mean, std = _band_constants(mean, std, ctx.device, "parse_shard")
        il, tl = _float_rows(int(idx["img_len"].max()) // esz, int(idx["tgt_len"].max()) // esz, num_classes)
        img_buf, tgt_buf = out if out is not None else (
            torch.empty((count, il), dtype=torch.float32, device=ctx.device),
            torch.empty((count, tl), dtype=torch.float32, device=ctx.device))
    sink = _make_sink(mode, verify_crc, img_buf, tgt_buf, mean, std, num_classes, channels)
    status = torch.empty((count,), dtype=torch.int32, device=ctx.device)
    isz = ctypes.sizeof(_lib.ExampleIndex)
    index_ptr = ctypes.c_void_p(si.index_dev.data_ptr() + first * isz) if si.index_dev is not None else None
    check(lib().b2_tfrecord_parse(
        ctx.handle, ptr(si.shard), si.nbytes, ctypes.c_void_p(si.rec_off.data_ptr() + 8 * first),
        ctypes.c_void_p(si.rec_len.data_ptr() + 8 * first), index_ptr, count,
        int(si.lens_host[first:first + count].max()), ctypes.byref(sink), ptr(status), ctx.stream()))
    return img_buf, tgt_buf, status


def example_layout(kind, img_bytes, tgt_bytes, img_h, img_w, img_c, tgt_h, tgt_w, identifier: bytes):
    """Host-side protobuf scaffold around the two payloads -> (scaffold bytes, piece_len[3], example_len)."""
    cap = 256 + len(identifier)
    buf = (ctypes.c_uint8 * cap)()
    pl = (ctypes.c_uint32 * 3)()
    el = ctypes.c_uint64()
    idb = (ctypes.c_uint8 * max(1, len(identifier))).from_buffer_copy(identifier or b"\0")
    check(lib().b2_example_layout(kind, int(img_bytes), int(tgt_bytes), int(img_h), int(img_w), int(img_c), int(tgt_h),
                                  int(tgt_w), ctypes.cast(idb, ctypes.c_void_p), len(identifier),
                                  ctypes.cast(buf, ctypes.c_void_p), cap, pl, ctypes.byref(el)))
    total = pl[0] + pl[1] + pl[2]
    return bytes(buf[:total]), (pl[0], pl[1], pl[2]), int(el.value)


class BuildPlan:
    """Descriptor tables of one batch of records, uploaded once; launch() enqueues the serialise + frame kernel."""

    def __init__(self, items, device=None):
        self.ctx = get_ctx(device)
        n = len(items)
        descs = np.zeros(n, dtype=np.dtype(_lib.BUILD_DESC_DTYPE))
        assert descs.dtype.itemsize == ctypes.sizeof(_lib.BuildDesc)
        scaf = bytearray()
        pos = 0
        self.offsets, self.keep = [], []
        max_rec = 0
        for i, it in enumerate(items):
            img, tgt, kind = it["img"], it["tgt"], int(it["kind"])
            self.keep += [img, tgt]
            ib = img.numel() * (img.element_size() if kind == 1 else 4)
            tb = tgt.numel() * (tgt.element_size() if kind == 1 else 4)
            sc, pl, el = example_layout(kind, ib, tb, it["h"], it["w"], it["c"], it["th"], it["tw"], it["identifier"])
            d = descs[i]
            d["out_off"], d["example_len"], d["scaffold_off"] = pos, el, len(scaf)
            d["piece_len"] = pl
            d["src_dtype"], d["tgt_dtype"], d["kind"] = b2_dtype(img), b2_dtype(tgt), kind
            d["img_src"], d["img_count"] = img.data_ptr(), img.numel() * (img.element_size() if kind == 1 else 1)
            d["tgt_src"], d["tgt_count"] = tgt.data_ptr(), tgt.numel() * (tgt.element_size() if kind == 1 else 1)
            scaf += sc
            self.offsets.append(pos)
            pos += el + 16
            max_rec = max(max_rec, el + 16)
        self.n, self.total, self.max_rec, self.itemsize = n, pos, max_rec, descs.dtype.itemsize
        self.out = torch.empty((_align16(pos) + 16,), dtype=torch.uint8, device=self.ctx.device)
        self.descs_d = to_device(descs.view(np.uint8), self.ctx.device)
        self.scaf_d = to_device(bytes(scaf) if scaf else b"\0", self.ctx.device)

    def launch(self):
        for s in range(0, self.n, 65535):
            m = min(65535, self.n - s)
            check(lib().b2_tfrecord_build(self.ctx.handle, ctypes.c_void_p(self.descs_d.data_ptr() + s * self.itemsize), m,
                                          self.max_rec, ptr(self.scaf_d), ptr(self.out), self.ctx.stream()))
        return self.out


def build_records(items, device=None):
    """Serialise + frame records on the device.

    items: list of dicts with keys img (CUDA tensor), tgt (CUDA tensor), kind (1 bytes / 2 float),
    h, w, c, th, tw, identifier (bytes).  Returns (out uint8 CUDA tensor holding the framed records back to
    back, offsets list, total bytes).
    """
    plan = BuildPlan(items, device)
    return plan.launch(), plan.offsets, plan.total


def _make_sink(mode, verify_crc, img_buf, tgt_buf, mean=None, std=None, num_classes=None, channels=None):
    """The b2_parse_sink for a mode; mean / std are float32 device tensors (their length is the band count).  The
    statistics modes take their band count from channels and their counters (or None) in img_buf / tgt_buf."""
    sink = _lib.ParseSink()
    sink.mode, esz = _sink_mode(mode)
    sink.verify_crc = 1 if verify_crc else 0
    if mode in _STATS_MODES:
        sink.img_out = img_buf.data_ptr() if img_buf is not None else None
        sink.tgt_out = tgt_buf.data_ptr() if tgt_buf is not None else None
        sink.channels = int(channels)
    elif mode == "raw":
        sink.img_out, sink.img_stride = img_buf.data_ptr(), img_buf.stride(0) * img_buf.element_size()
        sink.tgt_out, sink.tgt_stride = tgt_buf.data_ptr(), tgt_buf.stride(0) * tgt_buf.element_size()
    elif esz:
        sink.img_out, sink.img_stride = img_buf.data_ptr(), img_buf.stride(0) * 4
        sink.tgt_out, sink.tgt_stride = tgt_buf.data_ptr(), tgt_buf.stride(0) * 4
        sink.mean, sink.std = mean.data_ptr(), std.data_ptr()
        sink.channels, sink.num_classes = int(mean.numel()), int(num_classes)
        sink._keep = (mean, std)
    return sink


def parse_table(st: ShardTable, mode, img_elems=0, tgt_elems=0, verify_crc=True, mean=None, std=None, num_classes=None,
                out=None, status=None, want_img=True, want_tgt=True, channels=None):
    """Enqueue the fused pass over EVERY record of an opened shard; no host synchronisation.

    The record count lives on the device, so outputs are sized for st.max_records rows:
    mode 'raw': (max_records, img_elems) / (max_records, tgt_elems) uint8 rows of payload bytes as stored;
    mode 'norm_onehot' (uint8 BytesList records) and 'norm_onehot_f32' (packed float32 FloatList records):
    (max_records, img_elems) float32 and (max_records, tgt_elems*K) float32, sizes in elements (H*W*C and H*W);
    mode 'stats' / 'stats_f32': the (acc, hist) counters of parse_shard, added to out=(acc, hist) when given
    (img_elems / tgt_elems are not used);
    mode 'none': CRC verification only.  A payload longer than its row gives status 3.
    Returns (img_buf, tgt_buf, status_dev[max_records]); rows / entries >= the record count are untouched.
    """
    ctx = get_ctx(st.shard.device)
    cap = st.max_records
    _, esz = _sink_mode(mode)
    img_buf = tgt_buf = None
    if mode in _STATS_MODES:
        img_buf, tgt_buf = _stats_out(out, channels, ctx.device)
    elif mode == "raw":
        img_buf, tgt_buf = out if out is not None else (
            torch.empty((cap, _align16(max(1, img_elems))), dtype=torch.uint8, device=ctx.device),
            torch.empty((cap, _align16(max(1, tgt_elems))), dtype=torch.uint8, device=ctx.device))
    elif esz:
        mean, std = _band_constants(mean, std, ctx.device, "parse_table")
        il, tl = _float_rows(img_elems, tgt_elems, num_classes)
        img_buf, tgt_buf = out if out is not None else (
            torch.empty((cap, il), dtype=torch.float32, device=ctx.device),
            torch.empty((cap, tl), dtype=torch.float32, device=ctx.device))
    sink = _make_sink(mode, verify_crc, img_buf, tgt_buf, mean, std, num_classes, channels)
    if not want_img:
        sink.img_out = None          # the C ABI skips a NULL output
    if not want_tgt:
        sink.tgt_out = None
    if status is None:
        status = torch.empty((cap,), dtype=torch.int32, device=ctx.device)
    check(lib().b2_tfrecord_parse_table(ctx.handle, ptr(st.shard), st.nbytes, cap, ptr(st.table), ctypes.byref(sink),
                                        ptr(status), ctx.stream()))
    return img_buf, tgt_buf, status


class ShardPipeline:
    """Streams shards through upload -> open -> fused parse with NO per-shard host synchronisation.

    Two rings.  OPEN slots (`open_ahead` of them) own a device staging buffer (for host shards) and a shard table:
    upload + frame scan + feature index of later shards run ahead on high-priority streams — the fused pass is a
    persistent kernel that fills every SM, so the small open kernels can only run in the gaps between two fused
    passes and must be queued well before they are needed.  PARSE slots (`depth` of them) own the status array
    and the output buffers.  Iterating yields (img_buf, tgt_buf, status_dev, table) with the producing work already
    ordered before the caller's current stream; a parse slot is recycled `depth` shards later, after whatever
    the caller enqueued on its buffers.  In the statistics modes ('stats', 'stats_f32'; channels= bands) every slot adds
    into ONE (acc, hist) counter pair (self.stats_out, or out=), which each iteration yields as img_buf / tgt_buf.
    """

    def __init__(self, mode, img_elems, tgt_elems, max_records, verify_crc=True, mean=None, std=None, num_classes=None,
                 device=None, depth=3, max_shard_bytes=0, open_ahead=8, channels=None, out=None):
        self.ctx = get_ctx(device)
        dev = self.ctx.device
        self.mode, self.verify_crc, self.num_classes = mode, verify_crc, num_classes
        self.img_elems, self.tgt_elems, self.cap, self.depth = int(img_elems), int(tgt_elems), int(max_records), int(depth)
        self.open_ahead = max(int(open_ahead), self.depth)
        self.mean = self.std = None
        if mean is not None:
            self.mean, self.std = _band_constants(mean, std, dev, "ShardPipeline")
        self.open_streams = [torch.cuda.Stream(dev, priority=-1) for _ in range(min(self.open_ahead, 4))]
        self.streams = [torch.cuda.Stream(dev) for _ in range(self.depth)]
        self.oslots = [dict(stage=None, table=None, opened=torch.cuda.Event(), parsed=None) for _ in range(self.open_ahead)]
        self.ready = [torch.cuda.Event() for _ in range(self.depth)]
        self.release = [None] * self.depth
        self.channels = channels
        self.stats_out = _stats_out(out, int(channels), dev) if mode in _STATS_MODES else None
        self.slots = [dict(status=torch.zeros((self.cap,), dtype=torch.int32, device=dev), out=self.stats_out)
                      for _ in range(self.depth)]
        self.max_shard_bytes = int(max_shard_bytes)

    def reset_events(self):
        """Forget events of earlier passes (needed before the pipeline is recorded into a CUDA graph)."""
        self.release = [None] * self.depth
        for o in self.oslots:
            o["parsed"] = None

    def _submit_open(self, k, shard):
        o = self.oslots[k % self.open_ahead]
        ostream = self.open_streams[k % len(self.open_streams)]
        main = torch.cuda.current_stream(self.ctx.device)
        if o["parsed"] is not None:
            ostream.wait_event(o["parsed"])         # the fused pass that last read this table / staging buffer is done
        ostream.wait_stream(main)
        nbytes = int(shard.numel())
        with torch.cuda.stream(ostream):
            if not shard.is_cuda:
                if o["stage"] is None or o["stage"].numel() < nbytes:
                    o["stage"] = torch.empty((max(nbytes, self.max_shard_bytes) + 16,), dtype=torch.uint8, device=self.ctx.device)
                o["stage"][:nbytes].copy_(shard, non_blocking=True)
                shard = o["stage"]
            need = table_layout(nbytes, self.cap)[7]
            if o["table"] is None or o["table"].numel() < need:
                o["table"] = torch.empty((need + need // 8,), dtype=torch.uint8, device=self.ctx.device)
            st = open_shard_async(shard, self.ctx.device, self.cap, nbytes=nbytes, table=o["table"])
            o["opened"].record(ostream)
        return o, st

    def _submit_parse(self, k, opened):
        o, st = opened
        slot = k % self.depth
        sl, stream = self.slots[slot], self.streams[slot]
        if self.release[slot] is not None:
            stream.wait_event(self.release[slot])
        stream.wait_event(o["opened"])
        with torch.cuda.stream(stream):
            img, tgt, status = parse_table(st, self.mode, self.img_elems, self.tgt_elems, self.verify_crc, self.mean,
                                           self.std, self.num_classes, out=sl["out"], status=sl["status"],
                                           channels=self.channels)
            if sl["out"] is None and img is not None:
                sl["out"] = (img, tgt)
            self.ready[slot].record(stream)
            o["parsed"] = torch.cuda.Event()
            o["parsed"].record(stream)
        return slot, (img, tgt, status, st)

    def run(self, shards):
        main = torch.cuda.current_stream(self.ctx.device)
        it = iter(shards)
        opened, pending = [], []
        k_open = k_parse = 0
        exhausted = False
        while True:
            while not exhausted and len(opened) + len(pending) < self.open_ahead:
                try:
                    shard = next(it)
                except StopIteration:
                    exhausted = True
                    break
                opened.append(self._submit_open(k_open, shard))
                k_open += 1
            if opened and len(pending) < self.depth:
                pending.append(self._submit_parse(k_parse, opened.pop(0)))
                k_parse += 1
                continue
            if not pending:
                break
            slot, res = pending.pop(0)
            main.wait_event(self.ready[slot])
            yield res
            ev = torch.cuda.Event()
            ev.record(main)
            self.release[slot] = ev


class CapturedPass:
    """A whole pass over a fixed list of shards (device tensors or pinned host tensors) recorded as ONE CUDA graph:
    uploads, open, fused parse and the caller's per-shard consumer.  replay() enqueues everything with a single
    launch, so the host cost per shard disappears (the tables and kernels never needed the host in the first place)."""

    def __init__(self, pipe, shards, consume=None):
        self.pipe, self.shards = pipe, list(shards)
        for res in pipe.run(self.shards):               # warm-up: allocates every slot's buffers outside the capture
            if consume is not None:
                consume(*res)
        torch.cuda.synchronize(pipe.ctx.device)
        pipe.reset_events()                             # events recorded outside the capture must not leak into it
        self.graph = torch.cuda.CUDAGraph()
        self.results = []
        side = torch.cuda.Stream(pipe.ctx.device)
        side.wait_stream(torch.cuda.current_stream(pipe.ctx.device))
        l0 = pipe.ctx.launches
        with torch.cuda.stream(side):
            with torch.cuda.graph(self.graph, stream=side):
                for res in pipe.run(self.shards):
                    self.results.append(consume(*res) if consume is not None else res)
        self.launches_per_replay = pipe.ctx.launches - l0
        torch.cuda.current_stream(pipe.ctx.device).wait_stream(side)
        pipe.reset_events()

    def replay(self):
        self.graph.replay()
        return self.results


def iter_parsed_shards(shards, mode, verify_crc=True, mean=None, std=None, num_classes=None, out=None, device=None,
                       img_elems=None, tgt_elems=None, max_records=None, depth=3, channels=None):
    """Parse a sequence of shards (CUDA-resident or pinned-host uint8 tensors).

    With img_elems / tgt_elems / max_records given (the chip shape and records-per-shard bound a reader knows from
    its dataset), the shards stream through ShardPipeline without any host synchronisation.  Otherwise each shard
    is opened synchronously to learn its shapes.  Yields (img_buf, tgt_buf, status_dev, table-or-ShardIndex).
    The statistics modes take channels= and add every shard into one counter pair (out=, or new zeroed counters).
    """
    ctx = get_ctx(device)
    if img_elems is not None and max_records is not None:
        pipe = ShardPipeline(mode, img_elems, tgt_elems or 0, max_records, verify_crc, mean, std, num_classes, ctx.device, depth,
                             channels=channels, out=out)
        yield from pipe.run(shards)
        return
    if mode in _STATS_MODES:
        out = _stats_out(out, int(channels), ctx.device)
    for s in shards:
        si = open_shard(s, ctx.device)
        yield parse_shard(si, mode, verify_crc=verify_crc, mean=mean, std=std, num_classes=num_classes, out=out,
                          channels=channels) + (si,)


_STATS_KINDS = {"bytes": "stats", "float": "stats_f32"}


def shard_stats(shards, channels, kind="bytes", verify_crc=True, max_records=None, device=None, all_reduce=False):
    """Exact per-band image statistics and the label histogram of whole shards, each shard read once by the fused parse
    (b2chips.h B2_SINK_STATS / B2_SINK_STATS_F32).

    shards: CUDA-resident or pinned-host uint8 tensors (or bytes), streamed through ShardPipeline with no per-shard host
    synchronisation.  kind 'bytes': uint8 BytesList records; 'float': packed float32 FloatList records of integer values
    (uint8 / uint16 / int16 sources).  max_records bounds the records of one shard (default 4096).
    Returns (bands, histogram): bands = [(n, sum x, sum x^2)] exact Python ints per band, ready for mean_std_from_stats;
    histogram = 257 ints, bin v counting labels equal to v (0..255) and bin 256 every other label.
    Raises DataLossError when a frame, a data CRC or the feature template fails (the counters are then undefined), and
    B2Error when an image value of a 'float' shard is not an integer in [-2^16, 2^16).  With all_reduce=True and
    torch.distributed initialised, one all_reduce(SUM) of the packed integer counters (the failure counts included) gives
    every rank the same result, whatever the number of GPUs.  One device-to-host read, at the end.
    """
    if kind not in _STATS_KINDS:
        raise ValueError(kind)
    ctx = get_ctx(device)
    C, cap = int(channels), 4096 if max_records is None else int(max_records)
    src = [torch.from_numpy(np.frombuffer(s, np.uint8).copy()) if isinstance(s, (bytes, bytearray, memoryview)) else s
           for s in shards]
    pipe = ShardPipeline(_STATS_KINDS[kind], 0, 0, cap, verify_crc, device=ctx.device, channels=C,
                         max_shard_bytes=max((int(s.numel()) for s in src), default=0))
    # records with status != 0, shards with a bad frame, shards with more than cap records, shards
    tally = torch.zeros((4,), dtype=torch.int64, device=ctx.device)
    one = torch.ones((), dtype=torch.int64, device=ctx.device)
    for _, _, _, table in pipe.run(src):
        h = table.hdr_dev
        tally.add_(torch.stack((h[4], (h[1] == 1).long(), (h[1] == 2).long(), one)))
    acc, hist = pipe.stats_out
    packed = torch.cat((acc.reshape(-1), hist, tally))
    if all_reduce:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            t = packed if dist.get_backend() == "nccl" else packed.cpu()
            dist.all_reduce(t)                  # exact integer counters: the sum is the same in any order
            packed = t
    a = [int(x) for x in packed.cpu().numpy().view(np.uint64)]
    bad, frame, full, n_shards = a[-4:]
    if full:
        raise B2Error("%d shard(s) hold more than max_records=%d records" % (full, cap))
    if frame:
        raise DataLossError("corrupted record in %d shard(s) (bad frame or length CRC)" % frame)
    _check_bad_records(bad, "%d shard(s)" % n_shards)
    bands = []
    for c in range(C):
        n, sx, lo, hi, exc = a[5 * c:5 * c + 5]
        if exc:
            raise B2Error("shard_stats: band %d has %d value(s) that are not integers in [-65536, 65536)" % (c, exc))
        bands.append((n, sx - (1 << 64) if sx >> 63 else sx, lo + 65536 * hi))
    return bands, a[5 * C:5 * C + 257]


# ------------------------------------------------------------------------------------------------ label rasterisation
def project_points(xy, src_epsg, dst_epsg, device=None):
    """(N, 2) float64 vertices (NumPy or tensor) from one CRS to another -> (N, 2) float64 CUDA tensor.  b2_project_points.

    EPSG:4326 (longitude, latitude in degrees, GeoJSON axis order) and WGS84 UTM 326zz / 327zz, both ways and zone to zone;
    vertices the projection is not valid for come back as (NaN, NaN).  Raises B2Error for any other code.  Replaces the
    reprojection gdal.RasterizeLayer applies to each geometry (_descartes_img_chips.py:667-688)."""
    ctx = get_ctx(device)
    xy = to_device(xy, ctx.device)
    if xy.dtype != torch.float64 or xy.dim() != 2 or xy.shape[1] != 2:
        raise B2Error("project_points: expected (N, 2) float64 vertices, got %s %s" % (tuple(xy.shape), xy.dtype))
    out = torch.empty_like(xy)
    check(lib().b2_project_points(ctx.handle, ptr(xy), ptr(out), xy.shape[0], int(src_epsg), int(dst_epsg), ctx.stream()))
    return out


class RasterLayout:
    """The tables b2_rasterize_polygons reads, as NumPy arrays (include/b2chips.h): fill (E, 4) / fill_off, miny / job_off
    (one job per (feature, scanline)), job_ints_off (each job's room for its crossings), lines (L, 4) / line_feat, values."""

    def __init__(self, fill, fill_off, miny, job_off, job_ints_off, lines, line_feat, values):
        self.fill, self.fill_off, self.miny, self.job_off = fill, fill_off, miny, job_off
        self.job_ints_off, self.lines, self.line_feat, self.values = job_ints_off, lines, line_feat, values

    @property
    def n_jobs(self):
        return int(self.job_off[-1])


def rasterize_layout(features, size, all_touched=True):
    """The host half of rasterize_polygons (same arguments), on the CPU: lays the edges out and sizes the scanline
    workspace.  Raises B2Error for a burn value outside 0..255 or a non-finite vertex.

    A feature's scanlines are GDAL's [max((int) min y, 0), min((int) max y, H - 1)]; a feature whose y-range misses the
    raster has none.  A job's workspace is the number of the feature's non-horizontal edges whose y-span can hold its
    pixel-centre line (y_lo <= row + 0.5 < y_hi, widened by one row at each end), so it follows the crossings a scanline
    can have, not the size of the largest feature in the layer."""
    H, W = (int(size), int(size)) if np.isscalar(size) else (int(size[0]), int(size[1]))
    verts, vert_feat, fill, n_edges, ring_y, ring_feat, lines, line_feat, values = [], [], [], [], [], [], [], [], []
    for f, (rings, value) in enumerate(features):
        if not 0 <= int(value) <= 255:
            raise B2Error("rasterize_polygons: burn values must be 0..255 (GDT_Byte raster)")
        values.append(int(value))
        ne = 0
        for r in rings:
            r = np.asarray(r, dtype=np.float64).reshape(-1, 2)
            verts.append(r)
            vert_feat.append(np.full(len(r), f, np.int64))
            if len(r) < 2:
                continue
            ring_y.append(r[:, 1])
            ring_feat.append(f)
            closed = r[0, 0] == r[-1, 0] and r[0, 1] == r[-1, 1]
            o = r[:-1] if closed else r                          # fill: every vertex with its predecessor, wrapping around
            fill.append(np.concatenate([np.roll(o, 1, axis=0), o], axis=1))
            ne += len(o)
            if all_touched:                                      # edge walk: the ring as given (GDAL does not close it)
                lines.append(np.concatenate([r[:-1], r[1:]], axis=1))
                line_feat.append(np.full(len(r) - 1, f, np.uint32))
        n_edges.append(ne)
    nF = len(values)
    if verts:
        bad = ~np.isfinite(np.concatenate(verts)).all(axis=1)
        if bad.any():
            raise B2Error("rasterize_polygons: feature %d has a non-finite vertex"
                          % int(np.concatenate(vert_feat)[int(np.argmax(bad))]))
    # scanlines: (int) truncation of the feature's y-range, as GDAL's miny / maxy, clipped to the raster before any
    # integer conversion (a feature wholly above or below the raster, however far, has none)
    ymin, ymax = np.full(nF, np.inf), np.full(nF, -np.inf)
    if ring_y:
        np.minimum.at(ymin, ring_feat, [y.min() for y in ring_y])
        np.maximum.at(ymax, ring_feat, [y.max() for y in ring_y])
    lo, hi = np.clip(np.trunc(ymin), 0, H), np.clip(np.trunc(ymax), -1, H - 1)
    rows = np.maximum(hi - lo + 1, 0).astype(np.int64)
    miny = np.where(rows > 0, lo, 0).astype(np.int32)
    job_off = np.zeros(nF + 1, np.uint32)
    np.cumsum(rows, out=job_off[1:])
    n_jobs = int(job_off[-1])
    fill_a = np.ascontiguousarray(np.concatenate(fill)) if fill else np.zeros((0, 4))
    fill_off = np.zeros(nF + 1, np.uint32)
    np.cumsum(n_edges, out=fill_off[1:])
    # workspace: every non-horizontal edge adds one slot to each job whose row it can cross, counted in a difference
    # array over job indices
    fe = np.repeat(np.arange(nF), n_edges)
    y1, y2 = fill_a[:, 1], fill_a[:, 3]
    r0 = np.maximum(np.ceil(np.minimum(y1, y2) - 0.5) - 1, lo[fe])
    r1 = np.minimum(np.ceil(np.maximum(y1, y2) - 0.5), hi[fe])
    keep = (y1 != y2) & (r1 >= r0)
    start = job_off[fe[keep]].astype(np.int64) + (r0[keep] - lo[fe[keep]]).astype(np.int64)
    end = start + (r1[keep] - r0[keep]).astype(np.int64) + 1
    diff = np.bincount(start, minlength=n_jobs + 1) - np.bincount(end, minlength=n_jobs + 1)
    job_ints_off = np.zeros(n_jobs + 1, np.uint64)
    np.cumsum(np.cumsum(diff[:n_jobs]), out=job_ints_off[1:])
    line_a = np.ascontiguousarray(np.concatenate(lines)) if lines else np.zeros((0, 4))
    lf = np.concatenate(line_feat) if line_feat else np.zeros(0, np.uint32)
    return RasterLayout(fill_a, fill_off, miny, job_off, job_ints_off, line_a, lf, np.asarray(values, np.uint8))


def rasterize_polygons(features, size, background_value=255, all_touched=True, device=None):
    """Burn polygons into a (H, W) uint8 CUDA tensor with GDAL's RasterizeLayer semantics (ALL_TOUCHED by default).

    features: list of (rings, value) in burn order; rings = list of (N, 2) arrays in PIXEL space (x = column, y = line),
    first ring the shell, the others holes or further polygons (even-odd rule over all of them); value 0..255.
    Raises B2Error for a burn value outside 0..255 or a non-finite vertex, naming the feature.
    The host only lays the edges out (rasterize_layout, NumPy); the scanline fill, the edge walk and the last-feature-wins
    resolution run in b2_rasterize_polygons.  Replaces gdal.RasterizeLayer in create_label_array_for_tile
    (_descartes_img_chips.py:667-688)."""
    ctx = get_ctx(device)
    H, W = (int(size), int(size)) if np.isscalar(size) else (int(size[0]), int(size[1]))
    L = rasterize_layout(features, (H, W), all_touched)
    nF, n_jobs = len(L.values), L.n_jobs
    d = lambda a, dt: to_device(np.ascontiguousarray(a, dtype=dt).view(np.uint8).reshape(-1), ctx.device) if np.asarray(a).size else None
    fill_d, off_d, miny_d, job_d = d(L.fill, np.float64), d(L.fill_off, np.uint32), d(L.miny, np.int32), d(L.job_off, np.uint32)
    line_d, lf_d, val_d = d(L.lines, np.float64), d(L.line_feat, np.uint32), d(L.values, np.uint8)
    ints_off_d = d(L.job_ints_off, np.uint64) if n_jobs else None
    owner = torch.empty((H * W,), dtype=torch.int32, device=ctx.device)
    ints = torch.empty((max(1, int(L.job_ints_off[-1])),), dtype=torch.int32, device=ctx.device)
    out = torch.empty((H, W), dtype=torch.uint8, device=ctx.device)
    check(lib().b2_rasterize_polygons(ctx.handle, ptr(fill_d), ptr(off_d), ptr(miny_d), ptr(job_d), n_jobs, ptr(line_d), ptr(lf_d),
                                      len(L.line_feat), ptr(val_d), nF, W, H, int(background_value), ptr(ints_off_d), ptr(owner),
                                      ptr(ints), ptr(out), ctx.stream()))
    return out
