// tfrecord.cu — K2: TFRecord framing, CRC-32C, tf.train.Example payload location, fused payload kernels.
//
// Replaces (reference call sites): tf.io.TFRecordWriter.write  _img_to_tf_mp.py:119,141 / _img_to_tf_threaded.py:182,203
//                                   Example.SerializeToString   _img_to_tf_mp.py:141, convert_to_example
//                                                               _tfrecord_image_translation.py:160-211
//                                   TFRecordDataset reader      parse_tfrecords.ipynb cell 4
//                                   parse_single_example / decode_raw / reshape
//                                                               _tfrecord_image_translation.py:249,306-314,394-407
//
// Data layout: a shard is one contiguous device buffer.  The record CRC-32C is described in tfrecord_common.cuh.
#include <cstring>
#include <vector>

#include "tfrecord_common.cuh"

namespace b2 {

// ---------------------------------------------------------------------------------------------- scan
// Frames are a linked list (each length tells where the next header is), so the walk is inherently serial and,
// done naively, pays one cold HBM round trip (~1 us) per record.  Records of one shard have nearly the same
// length (fixed-size chips + a short identifier), so the CTA works in rounds of kScanR records:
//   1. all threads prefetch, with coalesced 128-bit loads, a window around the PREDICTED position of each of the
//      next kScanR headers (prediction = position of the current header + k * last stride),
//   2. thread 0 hops through shared memory: read 8 length bytes, add, next window — nothing else; the hop chain
//      ends at the first header that lies outside its window (the next round re-anchors there; the first window
//      of a round always contains its header, so every round advances),
//   3. one thread per visited header does what the hop skipped: bounds, capacity, masked length CRC (table in
//      shared memory, stored CRC from the window), and publishes offset / length; the first failure cuts the
//      walk exactly where RecordReader would stop.
// The result (record table, count, status) is identical to RecordReader's sequential walk for any input.
constexpr int kScanThreads = 512;
constexpr int kScanR = 128;
constexpr int kScanHW = 112;
constexpr int kScanWB = 2 * kScanHW + 32;   // bytes per window (multiple of 16)

// 8 bytes at an arbitrary byte offset of a 4-byte aligned shared-memory buffer: three word loads + two funnel shifts
__device__ __forceinline__ uint64_t smem_u64_unaligned(const uint8_t* base, uint32_t off) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(base) + (off >> 2);
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], sh = (off & 3) * 8;
    return (uint64_t)__funnelshift_r(w0, w1, sh) | ((uint64_t)__funnelshift_r(w1, w2, sh) << 32);
}

struct ScanOut {
    uint64_t* offs;
    uint64_t* lens;
    int64_t* hdr;          // [0] n, [1] status, [2] total tiles, [3] max len, [4] n_bad (zeroed here)
    uint32_t* tile_start;  // cap + 1 entries, or NULL (legacy b2_tfrecord_scan)
    unsigned long long* acc;   // cap entries zeroed here, or NULL
    int hdr_words;         // how many int64 of hdr exist (2 legacy, 8 table)
};

__global__ void __launch_bounds__(kScanThreads)
scan_kernel(const uint8_t* __restrict__ shard, uint64_t nbytes, uint64_t cap, ScanOut o,
            const CrcTables* __restrict__ tab) {
    __shared__ __align__(16) uint8_t win[kScanR][kScanWB + 16];
    __shared__ uint64_t w_lo[kScanR];            // absolute start of each window
    __shared__ uint64_t r_pos[kScanR];           // header positions visited this round
    __shared__ uint32_t s_crc[256];
    __shared__ uint64_t s_pos, s_est, s_n;
    __shared__ int s_m, s_state;                 // headers visited this round; 0 continue, 1 clean end, 2 error, 3 capacity
    __shared__ unsigned long long s_first_bad, s_maxlen;
    __shared__ int s_bad_kind;
    __shared__ uint32_t s_warp[kScanThreads / 32];
    const int tid = threadIdx.x;
    if (o.acc)
        for (uint64_t i = tid; i < cap; i += kScanThreads) o.acc[i] = 0ull;
    for (int i = tid; i < 256; i += kScanThreads) s_crc[i] = __ldg(&tab->t4[3][i]);
    if (tid == 0) {
        s_pos = 0;
        s_n = 0;
        s_est = 0;
        s_state = nbytes == 0 ? 1 : (nbytes < 12 ? 2 : 0);   // a shard shorter than one header is truncated
        s_maxlen = 0;
    }
    __syncthreads();
    while (s_state == 0) {
        const uint64_t base = s_pos, n0 = s_n;
        uint64_t est = s_est;
        if (est == 0) {                          // first round: learn the stride from the first header (1 round trip)
            if (tid == 0) {
                uint64_t e = 0;
                if (nbytes - base >= 12) {
                    const uint64_t l = rd_u64(shard + base);
                    if (l <= nbytes) e = l + 16;
                }
                s_est = e ? e : 16;
            }
            __syncthreads();
            est = s_est;
        }
        // 1. prefetch windows (vector kScanWB/16 of a window is slack for the unaligned 8-byte read)
        for (int i = tid; i < kScanR * (kScanWB / 16); i += kScanThreads) {
            const int k = i / (kScanWB / 16), j = i % (kScanWB / 16);
            const uint64_t c = base + (uint64_t)k * est;   // may overflow for a garbage est: harmless, only a prefetch hint
            const uint64_t lo = c > (uint64_t)kScanHW ? (c - kScanHW) & ~15ull : 0;
            if (j == 0) w_lo[k] = lo;
            const uint64_t a = lo + 16ull * j;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (a < nbytes && lo <= nbytes) v = ld16_bounded(shard, a, nbytes);
            reinterpret_cast<uint4*>(&win[k][0])[j] = v;
        }
        __syncthreads();
        // 2. serial hop chain over shared memory: nothing but "read length, add"
        if (tid == 0) {
            uint64_t pos = base;
            int m = 0;
            for (int k = 0; k < kScanR; k++) {
                const uint64_t off = pos - w_lo[k];                     // wraps to huge when pos < w_lo[k]
                if (off > (uint64_t)(kScanWB - 12) || pos >= nbytes || nbytes - pos < 12) break;
                const uint64_t l = smem_u64_unaligned(&win[k][0], (uint32_t)off);
                r_pos[m++] = pos;
                if (l > nbytes) break;                                  // certainly out of bounds: step 3 reports it
                pos += 16 + l;
            }
            s_m = m;
            s_first_bad = ~0ull;
            s_bad_kind = 0;
        }
        __syncthreads();
        // 3. everything the hop skipped, one thread per visited header, in RecordReader's order of checks
        const int m = s_m;
        for (int k = tid; k < m; k += kScanThreads) {
            const uint64_t pos = r_pos[k];
            const uint8_t* hp = &win[k][pos - w_lo[k]];
            const uint64_t l = rd_u64(hp);
            const bool crc_bad = crc_hdr8(l, s_crc) != rd_u32(hp + 8);
            const bool bounds_bad = l > nbytes - pos - 12 || nbytes - pos - 12 - l < 4;
            const bool cap_bad = n0 + k >= cap;
            if (crc_bad || bounds_bad || cap_bad) {
                atomicMin(&s_first_bad, (unsigned long long)k);
            } else {
                o.offs[n0 + k] = pos + 12;
                o.lens[n0 + k] = l;
            }
        }
        __syncthreads();
        if (tid == 0) {
            const unsigned long long fb = s_first_bad;
            if (fb != ~0ull) {                   // the walk stops at header fb of this round
                const uint64_t pos = r_pos[fb];
                const uint8_t* hp = &win[fb][pos - w_lo[fb]];
                const uint64_t l = rd_u64(hp);
                const bool crc_bad = crc_hdr8(l, s_crc) != rd_u32(hp + 8);
                const bool bounds_bad = l > nbytes - pos - 12 || nbytes - pos - 12 - l < 4;
                s_n = n0 + fb;
                s_state = (crc_bad || bounds_bad) ? 2 : 3;
            } else {
                s_n = n0 + m;
                const uint64_t last = r_pos[m - 1];
                const uint64_t l = rd_u64(&win[m - 1][last - w_lo[m - 1]]);
                const uint64_t pos = last + 16 + l;      // in bounds: header m-1 passed the checks
                s_pos = pos;
                s_est = 16 + l;
                if (pos >= nbytes) s_state = 1;          // == nbytes: clean end
                else if (nbytes - pos < 12) s_state = 2; // truncated header
            }
        }
        __syncthreads();
    }
    const uint64_t n = s_n;
    const int64_t st = s_state == 1 ? 0 : (s_state == 3 ? 2 : 1);
    if (tid == 0) {
        o.hdr[0] = (int64_t)n;
        o.hdr[1] = st;
    }
    if (o.hdr_words < 5) return;
    // tile prefix over the n records (records past a corruption are not counted)
    uint64_t maxlen = 0;
    const uint32_t per = (uint32_t)((n + kScanThreads - 1) / kScanThreads);
    const uint64_t k0 = (uint64_t)tid * per, k1 = (k0 + per < n) ? k0 + per : n;
    uint32_t sum = 0;
    for (uint64_t k = k0; k < k1; k++) {
        const uint64_t l = o.lens[k];
        sum += record_tiles(o.offs[k], l);
        maxlen = l > maxlen ? l : maxlen;
    }
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if ((tid & 31) >= d) inc += t;
    }
    if ((tid & 31) == 31) s_warp[tid >> 5] = inc;
    __syncthreads();
    uint32_t wbase = 0;
    for (int w = 0; w < (tid >> 5); w++) wbase += s_warp[w];
    uint32_t run = wbase + inc - sum;
    for (uint64_t k = k0; k < k1; k++) {
        o.tile_start[k] = run;
        run += record_tiles(o.offs[k], o.lens[k]);
    }
    atomicMax(&s_maxlen, (unsigned long long)maxlen);
    __syncthreads();
    if (tid == kScanThreads - 1) {
        o.tile_start[n] = run;
        o.hdr[2] = (int64_t)run;
        o.hdr[3] = (int64_t)s_maxlen;
        o.hdr[4] = 0;
        o.hdr[5] = 0;   // chunk scheduler words of the fused pass
    }
}

// ---------------------------------------------------------------------------------------------- index
// One WARP per record walks the protobuf structure (SURVEY.md App. A) in two phases:
//   A. all lanes together hop over the map entries of Example.features (tag + length, then skip), reading through
//      a 512-byte window of the shard in shared memory that the warp refills with one coalesced 128-bit load per
//      lane — a record costs a handful of HBM round trips (entry headers sit in three clusters: before the image
//      payload, between the payloads, after the target payload), not one per byte;
//   B. lane e then parses entry e on its own (key, Feature oneof, list, value) through a private 128-byte window,
//      so the eight entries of a record are decoded side by side instead of one after the other;
//   C. lane 0 applies the per-entry results in file order (last duplicate wins, like a protobuf map).
// Everything is bounds-checked against the record; a malformed message sets status 1 instead of faulting.
constexpr int kIdxWarps = 4;
constexpr int kIdxWin = 512;    // phase A window, per warp
constexpr int kLaneWin = 128;   // phase B window, per lane
struct Win {
    const uint8_t* g;
    uint64_t nbytes;   // bytes that may be read from g
    uint8_t* s;        // shared-memory backing
    uint64_t lo;       // window = [lo, lo + size)
};
__device__ __forceinline__ uint32_t win_byte(Win& w, uint64_t p) {   // warp-uniform p: cooperative refill
    if (p - w.lo >= (uint64_t)kIdxWin) {
        __syncwarp();
        w.lo = p & ~15ull;
        const uint64_t a = w.lo + 16ull * (threadIdx.x & 31);
        uint4 v = make_uint4(0, 0, 0, 0);
        if (a < w.nbytes) v = ld16_bounded(w.g, a, w.nbytes);
        reinterpret_cast<uint4*>(w.s)[threadIdx.x & 31] = v;
        __syncwarp();
    }
    return w.s[p - w.lo];
}
__device__ __forceinline__ uint32_t lane_byte(Win& w, uint64_t p) {  // per-lane p: private refill
    if (p - w.lo >= (uint64_t)kLaneWin) {
        w.lo = p & ~15ull;
#pragma unroll
        for (int j = 0; j < kLaneWin / 16; j++) {
            const uint64_t a = w.lo + 16ull * j;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (a < w.nbytes) v = ld16_bounded(w.g, a, w.nbytes);
            reinterpret_cast<uint4*>(w.s)[j] = v;
        }
    }
    return w.s[p - w.lo];
}
struct Cursor {
    uint64_t p, end;
    bool ok;
};
template <bool kLane>
__device__ __forceinline__ uint32_t rd_byte(Win& w, uint64_t p) { return kLane ? lane_byte(w, p) : win_byte(w, p); }
template <bool kLane>
__device__ inline uint64_t rd_varint(Win& w, Cursor& c) {
    uint64_t v = 0;
    for (int s = 0; s < 70; s += 7) {
        if (c.p >= c.end) { c.ok = false; return 0; }
        const uint32_t x = rd_byte<kLane>(w, c.p++);
        v |= (uint64_t)(x & 0x7F) << s;
        if (!(x & 0x80)) return v;
    }
    c.ok = false;
    return 0;
}
// reads a tag and, for LEN fields, the sub-range; skips other wire types. returns field number (0 on end/error)
template <bool kLane>
__device__ inline uint32_t next_field(Win& w, Cursor& c, int& wt, uint64_t& v0, uint64_t& v1) {
    if (!c.ok || c.p >= c.end) return 0;
    const uint64_t tag = rd_varint<kLane>(w, c);
    if (!c.ok) return 0;
    wt = (int)(tag & 7);
    const uint32_t f = (uint32_t)(tag >> 3);
    if (wt == 0) {
        v0 = rd_varint<kLane>(w, c);
    } else if (wt == 1) {
        v0 = c.p; v1 = c.p + 8; c.p += 8;
    } else if (wt == 5) {
        v0 = c.p; v1 = c.p + 4; c.p += 4;
    } else if (wt == 2) {
        const uint64_t n = rd_varint<kLane>(w, c);
        if (!c.ok || n > c.end - c.p) { c.ok = false; return 0; }
        v0 = c.p; v1 = c.p + n; c.p += n;
    } else {
        c.ok = false;
        return 0;
    }
    if (c.p > c.end) { c.ok = false; return 0; }
    if (f == 0) { c.ok = false; return 0; }
    return f;
}
__device__ inline bool key_is(Win& w, uint64_t s, uint64_t e, const char* lit, int n) {
    if (e - s != (uint64_t)n) return false;
    for (int i = 0; i < n; i++)
        if (lane_byte(w, s + i) != (uint32_t)(uint8_t)lit[i]) return false;
    return true;
}

struct EntryResult {     // what one map entry contributes
    uint64_t ps, pe;     // payload / identifier byte range
    int64_t ival;
    int32_t which;       // 0 img, 1 h, 2 w, 3 c, 4 tgt, 5 th, 6 tw, 7 id; -1 not ours; -2 malformed
    int32_t okk;         // payload kind (1 bytes, 2 floats) or 1 = well-formed scalar, 0 = wrong type / count
};

// phase B: parse ONE map entry [a2, b2v)
__device__ inline EntryResult parse_entry(Win& w, uint64_t a2, uint64_t b2v) {
    EntryResult r;
    r.ps = r.pe = 0; r.ival = 0; r.which = -1; r.okk = 0;
    Cursor en{a2, b2v, true};
    int wt3; uint64_t a3, b3;
    uint64_t ks = 0, ke = 0, vs = 0, ve = 0;
    bool hk = false, hv = false;
    while (uint32_t f3 = next_field<true>(w, en, wt3, a3, b3)) {
        if (f3 == 1 && wt3 == 2) { ks = a3; ke = b3; hk = true; }
        else if (f3 == 2 && wt3 == 2) { vs = a3; ve = b3; hv = true; }
    }
    if (!en.ok) { r.which = -2; return r; }
    if (!hk) return r;
    int which = -1;
    if (key_is(w, ks, ke, "image/image_data", 16)) which = 0;
    else if (key_is(w, ks, ke, "image/height", 12)) which = 1;
    else if (key_is(w, ks, ke, "image/width", 11)) which = 2;
    else if (key_is(w, ks, ke, "image/channels", 14)) which = 3;
    else if (key_is(w, ks, ke, "target/target_data", 18)) which = 4;
    else if (key_is(w, ks, ke, "target/height", 13)) which = 5;
    else if (key_is(w, ks, ke, "target/width", 12)) which = 6;
    else if (key_is(w, ks, ke, "identifier", 10)) which = 7;
    if (which < 0) return r;
    // Feature oneof: last member present wins
    int kind = 0; uint64_t ls = 0, le = 0;
    if (hv) {
        Cursor fe{vs, ve, true};
        int wt4; uint64_t a4, b4;
        while (uint32_t f4 = next_field<true>(w, fe, wt4, a4, b4)) {
            if (wt4 == 2 && f4 >= 1 && f4 <= 3) { kind = (int)f4; ls = a4; le = b4; }
        }
        if (!fe.ok) { r.which = -2; return r; }
    }
    // the list message: field 1 repeated
    uint64_t ps = 0, pe = 0; int count = 0; int64_t ival = 0; bool packed_ok = true;
    if (kind) {
        Cursor li{ls, le, true};
        int wt5; uint64_t a5, b5;
        while (uint32_t f5 = next_field<true>(w, li, wt5, a5, b5)) {
            if (f5 != 1) continue;
            if (kind == 1) {
                if (wt5 == 2) { ps = a5; pe = b5; count++; }
            } else if (kind == 2) {
                if (wt5 == 2) { ps = a5; pe = b5; count++; }      // packed floats (one chunk expected)
                else if (wt5 == 5) { packed_ok = false; }          // unpacked fixed32: not supported on device
            } else {
                if (wt5 == 2) {
                    Cursor pk{a5, b5, true};
                    while (pk.ok && pk.p < pk.end) { ival = (int64_t)rd_varint<true>(w, pk); count++; }
                    if (!pk.ok) li.ok = false;
                } else if (wt5 == 0) { ival = (int64_t)a5; count++; }
            }
        }
        if (!li.ok) { r.which = -2; return r; }
    }
    r.which = which;
    r.ps = ps; r.pe = pe; r.ival = ival;
    if (which == 0 || which == 4) {
        if (kind == 1 && count == 1) r.okk = 1;
        else if (kind == 2 && packed_ok && count <= 1 && ((pe - ps) & 3) == 0) r.okk = 2;
    } else if (which == 7) {
        r.okk = (kind == 1 && count == 1) ? 1 : 0;
    } else {
        r.okk = (kind == 3 && count == 1) ? 1 : 0;
    }
    return r;
}

__global__ void __launch_bounds__(kIdxWarps * 32)
index_kernel(const uint8_t* __restrict__ shard, uint64_t nbytes, const uint64_t* __restrict__ rec_off,
             const uint64_t* __restrict__ rec_len, int n, b2_example_index* __restrict__ out,
             const int64_t* __restrict__ n_dev, const uint32_t* __restrict__ tile_start, uint32_t* __restrict__ tile2rec) {
    __shared__ __align__(16) uint8_t s_win[kIdxWarps][kIdxWin];
    __shared__ __align__(16) uint8_t s_lane[kIdxWarps][32][kLaneWin];
    __shared__ uint64_t s_ent[kIdxWarps][32][2];
    __shared__ EntryResult s_res[kIdxWarps][32];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * kIdxWarps + wib;
    if (n_dev && (int64_t)r >= n_dev[0]) return;   // opened shard: the record count is only known on the device
    if (r >= n) return;
    const uint64_t d0 = rec_off[r], dl = rec_len[r];
    if (tile2rec) {
        const uint32_t t0 = tile_start[r], t1 = tile_start[r + 1];
        for (uint32_t t = t0 + lane; t < t1; t += 32) tile2rec[t] = (uint32_t)r;
    }
    const uint64_t lim = nbytes < d0 + dl ? nbytes : d0 + dl;
    Win w{shard, lim, &s_win[wib][0], ~0ull - kIdxWin};
    Win lw{shard, lim, &s_lane[wib][lane][0], ~0ull - kLaneWin};
    b2_example_index ix;
    memset(&ix, 0, sizeof(ix));
    int have[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // img, h, w, c, tgt, th, tw, id : 1 ok, -1 wrong type/count
    int64_t dims[5] = {0, 0, 0, 0, 0};
    bool ok = true;
    Cursor ex{d0, d0 + dl, true};
    int wt; uint64_t a, b;
    while (uint32_t f = next_field<false>(w, ex, wt, a, b)) {
        if (f != 1 || wt != 2) continue;  // Example.features
        Cursor fs{a, b, true};
        bool more = true;
        while (more && ok) {
            // phase A: collect up to 32 map entries
            int ne = 0;
            int wt2; uint64_t a2, b2v;
            while (ne < 32) {
                const uint32_t f2 = next_field<false>(w, fs, wt2, a2, b2v);
                if (!f2) { more = false; break; }
                if (f2 != 1 || wt2 != 2) continue;  // Features.feature map entry
                if (lane == 0) { s_ent[wib][ne][0] = a2; s_ent[wib][ne][1] = b2v; }
                ne++;
            }
            if (!fs.ok) { ok = false; break; }
            __syncwarp();
            // phase B: one entry per lane
            if (lane < ne) s_res[wib][lane] = parse_entry(lw, s_ent[wib][lane][0], s_ent[wib][lane][1]);
            __syncwarp();
            // phase C: apply in file order (all lanes redundantly: the state stays warp-uniform)
            for (int e = 0; e < ne; e++) {
                const EntryResult q = s_res[wib][e];
                if (q.which == -2) { ok = false; break; }
                if (q.which < 0) continue;
                if (q.which == 0) { ix.img_off = q.ps; ix.img_len = q.pe - q.ps; ix.img_kind = q.okk; have[0] = q.okk ? 1 : -1; }
                else if (q.which == 4) { ix.tgt_off = q.ps; ix.tgt_len = q.pe - q.ps; ix.tgt_kind = q.okk; have[4] = q.okk ? 1 : -1; }
                else if (q.which == 7) {
                    if (q.okk) { ix.id_off = q.ps; ix.id_len = q.pe - q.ps; have[7] = 1; } else have[7] = -1;
                } else {
                    const int d = q.which < 4 ? q.which - 1 : q.which - 2;  // h,w,c,th,tw -> 0..4
                    if (q.okk) { dims[d] = q.ival; have[q.which] = 1; } else have[q.which] = -1;
                }
            }
            __syncwarp();
        }
        if (!ok) break;
    }
    if (!ex.ok) ok = false;
    ix.height = (int32_t)dims[0]; ix.width = (int32_t)dims[1]; ix.channels = (int32_t)dims[2];
    ix.tgt_height = (int32_t)dims[3]; ix.tgt_width = (int32_t)dims[4];
    int st = ok ? 0 : 1;
    if (st == 0)
        for (int k = 0; k < 8; k++)
            if (have[k] != 1) st = 2;
    ix.status = st;
    if (lane == 0) out[r] = ix;
}

// ---------------------------------------------------------------------------------------------- build
struct BuildArgs {
    const b2_build_desc* descs;
    const uint8_t* scaffold;
    uint8_t* out;
    const CrcTables* tab;
    unsigned long long* acc;   // per record { CRC partial, tiles done }, zero on entry
};

__device__ __forceinline__ uint32_t elem_as_f32_bits(const void* src, int dtype, uint64_t i, uint64_t count) {
    if (i >= count) return 0;
    float f;
    switch (dtype) {
        case B2_U8: f = (float)static_cast<const uint8_t*>(src)[i]; break;
        case B2_I8: f = (float)static_cast<const int8_t*>(src)[i]; break;
        case B2_U16: f = (float)static_cast<const uint16_t*>(src)[i]; break;
        case B2_I16: f = (float)static_cast<const int16_t*>(src)[i]; break;
        case B2_U32: f = (float)static_cast<const uint32_t*>(src)[i]; break;
        case B2_I32: f = (float)static_cast<const int32_t*>(src)[i]; break;
        case B2_F32: f = static_cast<const float*>(src)[i]; break;
        default: f = (float)static_cast<const double*>(src)[i]; break;
    }
    return __float_as_uint(f);
}

// byte j of a payload
__device__ __forceinline__ uint32_t payload_byte(const void* src, int kind, int dtype, uint64_t j, uint64_t count) {
    if (kind == 1) return static_cast<const uint8_t*>(src)[j];
    return (elem_as_f32_bits(src, dtype, j >> 2, count) >> (8 * (j & 3))) & 0xFFu;
}
// four consecutive payload bytes j..j+3 (all inside the payload)
__device__ __forceinline__ uint32_t payload_word(const void* src, int kind, int dtype, uint64_t j, uint64_t count) {
    if (kind == 1) {
        const uint8_t* p = static_cast<const uint8_t*>(src) + j;
        if ((reinterpret_cast<uintptr_t>(p) & 3) == 0) return *reinterpret_cast<const uint32_t*>(p);
        const uint32_t* q = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~uintptr_t(3));
        const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3) * 8;
        // the second aligned word may lie past the payload end only if j+4 == count and p unaligned: then its
        // needed bytes are still inside, so the aligned read stays within the allocation's last word
        return __funnelshift_r(q[0], q[1], sh);
    }
    const uint32_t b0 = elem_as_f32_bits(src, dtype, j >> 2, count);
    if ((j & 3) == 0) return b0;
    const uint32_t b1 = elem_as_f32_bits(src, dtype, (j >> 2) + 1, count);
    return __funnelshift_r(b0, b1, (uint32_t)(j & 3) * 8);
}

constexpr int kBuildRun = 4;   // consecutive tiles of one record per CTA: tables, header CRC and the per-thread CRC
                               // alignment are paid once per run

__global__ void __launch_bounds__(kTileThreads, 8) build_kernel(const BuildArgs a) {
    __shared__ __align__(16) uint4 buf4[kTile / 16];
    __shared__ CrcSmem cs;
    __shared__ uint32_t red[kTileThreads / 32];
    __shared__ uint32_t hdr_crc;
    const int r = blockIdx.y;
    const b2_build_desc d = a.descs[r];
    const uint64_t rs = d.out_off, L = d.example_len;
    const uint64_t d0 = rs + 12, d1 = d0 + L, re = d1;  // footer (4 bytes at d1) is written by whoever completes the record
    const uint64_t A = rs & ~15ull;
    const uint32_t t_end = (uint32_t)((re - A + kTile - 1) / kTile);        // tiles of this record (L == 0: header only)
    const uint32_t t_lo = blockIdx.x * kBuildRun;
    if (t_lo >= t_end) return;
    const uint32_t t_hi = t_lo + kBuildRun < t_end ? t_lo + kBuildRun : t_end;
    load_crc_tables(&cs, a.tab);
    if (threadIdx.x == 0) hdr_crc = crc_hdr8(L, a.tab->t4[3]);
    __syncthreads();
    uint32_t crc_state = 0;                                              // this thread's running CRC over the run
  for (uint32_t tile = t_lo; tile < t_hi; tile++) {
    const uint64_t ts = A + (uint64_t)tile * kTile, te = ts + kTile;
    const uint64_t ib = d.kind == 1 ? d.img_count : d.img_count * 4, tb = d.kind == 1 ? d.tgt_count : d.tgt_count * 4;
    // Example-space segment boundaries
    const uint64_t e1 = d.piece_len[0], e2 = e1 + ib, e3 = e2 + d.piece_len[1], e4 = e3 + tb;
    const uint8_t* sc = a.scaffold + d.scaffold_off;
    uint32_t* buf32 = reinterpret_cast<uint32_t*>(buf4);
    // Fast path: the whole tile lies inside ONE payload (31 of the 33 tiles of a cfg1 record).  Its bytes are then a
    // plain copy (BytesList) or a widening to float32 (FloatList) of a contiguous source range at an arbitrary byte
    // phase: each thread produces 16 tile bytes from two aligned source vectors and a funnel shift.
    {
        const int64_t e_lo = (int64_t)ts - (int64_t)d0, e_hi = (int64_t)te - (int64_t)d0;
        const void* psrc = nullptr;
        uint64_t pstart = 0, pcount = 0;
        int pdtype = 0;
        if (e_lo >= (int64_t)e1 && (uint64_t)e_hi <= e2) { psrc = d.img_src; pstart = (uint64_t)e_lo - e1; pcount = d.img_count; pdtype = d.src_dtype; }
        else if (e_lo >= (int64_t)e3 && (uint64_t)e_hi <= e4) { psrc = d.tgt_src; pstart = (uint64_t)e_lo - e3; pcount = d.tgt_count; pdtype = d.tgt_dtype; }
        if (psrc && d.kind == 1 && (reinterpret_cast<uintptr_t>(psrc) & 3) == 0) {
            // payload bytes [pstart, pstart + kTile) -> tile; source words are 4-byte aligned, phase = pstart & 3
            const uint32_t* q = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(psrc) + (pstart & ~3ull));
            const uint32_t sh = (uint32_t)(pstart & 3) * 8;
            const uint64_t last_word = (pcount + 3) / 4 - 1 - (pstart >> 2);   // last source word that may be read
            for (int g = threadIdx.x; g < kTile / 16; g += blockDim.x) {
                uint32_t wv[5];
#pragma unroll
                for (int k = 0; k < 5; k++) {
                    const uint64_t wi = 4ull * g + k;
                    wv[k] = (wi <= last_word && (k < 4 || sh)) ? __ldg(q + wi) : 0u;
                }
                buf4[g] = make_uint4(__funnelshift_r(wv[0], wv[1], sh), __funnelshift_r(wv[1], wv[2], sh),
                                     __funnelshift_r(wv[2], wv[3], sh), __funnelshift_r(wv[3], wv[4], sh));
            }
            goto staged;
        }
        if (psrc && d.kind == 2 && (pdtype == B2_U16 || pdtype == B2_U8)) {
            // payload bytes = float32(element i) little-endian; tile starts at payload byte pstart (phase pstart & 3)
            const uint64_t i0 = pstart >> 2;
            const uint32_t sh = (uint32_t)(pstart & 3) * 8;
            for (int w = threadIdx.x; w < kTile / 4; w += blockDim.x) {
                const uint64_t i = i0 + w;
                uint32_t a, b;
                if (pdtype == B2_U16) {
                    a = i < pcount ? __float_as_uint((float)__ldg(static_cast<const uint16_t*>(psrc) + i)) : 0u;
                    b = (sh && i + 1 < pcount) ? __float_as_uint((float)__ldg(static_cast<const uint16_t*>(psrc) + i + 1)) : 0u;
                } else {
                    a = i < pcount ? __float_as_uint((float)__ldg(static_cast<const uint8_t*>(psrc) + i)) : 0u;
                    b = (sh && i + 1 < pcount) ? __float_as_uint((float)__ldg(static_cast<const uint8_t*>(psrc) + i + 1)) : 0u;
                }
                buf32[w] = __funnelshift_r(a, b, sh);
            }
            goto staged;
        }
    }
    for (int w = threadIdx.x; w < kTile / 4; w += blockDim.x) {
        const uint64_t p = ts + 4ull * w;  // absolute position of this word
        uint32_t word = 0;
        if (p + 4 > rs && p < re) {
            const int64_t e = (int64_t)p - (int64_t)d0;  // Example-space offset of byte 0
            if (e >= (int64_t)e1 && (uint64_t)e + 4 <= e2) {
                word = payload_word(d.img_src, d.kind, d.src_dtype, (uint64_t)e - e1, d.img_count);
            } else if (e >= (int64_t)e3 && (uint64_t)e + 4 <= e4) {
                word = payload_word(d.tgt_src, d.kind, d.tgt_dtype, (uint64_t)e - e3, d.tgt_count);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const uint64_t q = p + j;
                    if (q < rs || q >= re) continue;
                    uint32_t bv;
                    const uint64_t rel = q - rs;
                    if (rel < 8) bv = (uint32_t)((L >> (8 * rel)) & 0xFF);
                    else if (rel < 12) bv = (hdr_crc >> (8 * (rel - 8))) & 0xFF;
                    else {
                        const uint64_t x = rel - 12;
                        if (x < e1) bv = sc[x];
                        else if (x < e2) bv = payload_byte(d.img_src, d.kind, d.src_dtype, x - e1, d.img_count);
                        else if (x < e3) bv = sc[e1 + (x - e2)];
                        else if (x < e4) bv = payload_byte(d.tgt_src, d.kind, d.tgt_dtype, x - e3, d.tgt_count);
                        else bv = sc[e1 + d.piece_len[1] + (x - e4)];
                    }
                    word |= bv << (8 * j);
                }
            }
        }
        buf32[w] = word;
    }
staged:
    __syncthreads();
    // write out the bytes of [max(ts,rs), min(te,re))
    const uint8_t* buf8 = reinterpret_cast<const uint8_t*>(buf4);
    for (int k = threadIdx.x; k < kTile / 16; k += blockDim.x) {
        const uint64_t p = ts + 16ull * k;
        if (p >= rs && p + 16 <= re) {
            st_cs(reinterpret_cast<uint4*>(a.out + p), buf4[k]);
        } else if (p + 16 > rs && p < re) {
            for (int j = 0; j < 16; j++)
                if (p + j >= rs && p + j < re) a.out[p + j] = buf8[16 * k + j];
        }
    }
    // running CRC over the data range; the tile grid is anchored at A = rs & ~15
    if (crc_tiled(L) && te > d0) crc_state = crc_running_step(crc_state, buf4, &cs, ts, d0, d1, ts <= d0 && d0 < te, ts >= d0 && te <= d1);
    __syncthreads();                                                       // buf4 is restaged by the next tile
  }
    // End of the run: fold the threads' states (a record too short for a partial leaves them zero) and merge the run into
    // the record's accumulator; the CTA that completes the record writes the masked CRC footer.
    const uint32_t t = crc_lane_partial(a.tab, crc_state);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t c = 0;
#pragma unroll
        for (int k = 0; k < kTileThreads / 32; k++) c ^= red[k];
        const unsigned long long upd = record_acc_merge(a.tab, a.acc + r, c, t_end - t_hi, t_hi - t_lo);
        if ((uint32_t)(upd >> 32) == t_end) {
            // an Example shorter than 4 bytes has no payload: its bytes are scaffold bytes
            const uint32_t m = mask_crc(record_crc(a.tab, (uint32_t)upd, A + (uint64_t)t_end * kTile - d1,
                                                   a.scaffold + d.scaffold_off, L));
            for (int j = 0; j < 4; j++) a.out[d1 + j] = (uint8_t)(m >> (8 * j));
        }
    }
}

}  // namespace b2

using namespace b2;

extern "C" int b2_tfrecord_scan(b2_ctx* ctx, const uint8_t* shard, uint64_t nbytes, uint64_t max_records,
                                uint64_t* rec_off, uint64_t* rec_len, int64_t* result, b2_stream stream) {
    B2_REQUIRE(ctx && (shard || nbytes == 0) && rec_off && rec_len && result, "b2_tfrecord_scan: NULL argument");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(shard) & 15) == 0, "b2_tfrecord_scan: shard must be 16-byte aligned");
    DeviceGuard g(ctx->device);
    ScanOut o{rec_off, rec_len, result, nullptr, nullptr, 2};
    scan_kernel<<<1, kScanThreads, 0, static_cast<cudaStream_t>(stream)>>>(shard, nbytes, max_records, o, ctx->crc_dev);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int b2_tfrecord_index(b2_ctx* ctx, const uint8_t* shard, const uint64_t* rec_off, const uint64_t* rec_len,
                                 int n, b2_example_index* out, b2_stream stream) {
    B2_REQUIRE(ctx && shard && rec_off && rec_len && out, "b2_tfrecord_index: NULL argument");
    B2_REQUIRE(n >= 0, "b2_tfrecord_index: n < 0");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(shard) & 15) == 0, "b2_tfrecord_index: shard must be 16-byte aligned");
    if (n == 0) return 0;
    DeviceGuard g(ctx->device);
    index_kernel<<<(n + kIdxWarps - 1) / kIdxWarps, kIdxWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        shard, ~0ull, rec_off, rec_len, n, out, nullptr, nullptr, nullptr);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

extern "C" uint64_t b2_tfrecord_table_bytes(uint64_t shard_nbytes, uint64_t max_records) {
    return table_bytes(shard_nbytes, max_records);
}

extern "C" int b2_tfrecord_table_layout(uint64_t shard_nbytes, uint64_t max_records, uint64_t offsets[8]) {
    B2_REQUIRE(offsets, "b2_tfrecord_table_layout: NULL argument");
    B2_REQUIRE(max_records >= 1 && max_records <= (1u << 24), "b2_tfrecord_table_layout: max_records out of range");
    const TableView v = table_view(nullptr, shard_nbytes, max_records);
    offsets[0] = reinterpret_cast<uintptr_t>(v.hdr);
    offsets[1] = reinterpret_cast<uintptr_t>(v.rec_off);
    offsets[2] = reinterpret_cast<uintptr_t>(v.rec_len);
    offsets[3] = reinterpret_cast<uintptr_t>(v.index);
    offsets[4] = reinterpret_cast<uintptr_t>(v.tile_start);
    offsets[5] = reinterpret_cast<uintptr_t>(v.tile2rec);
    offsets[6] = v.cap_tiles;
    offsets[7] = table_bytes(shard_nbytes, max_records);
    return 0;
}

extern "C" int b2_tfrecord_open(b2_ctx* ctx, const uint8_t* shard, uint64_t nbytes, uint64_t max_records, uint8_t* table,
                                b2_stream stream) {
    B2_REQUIRE(ctx && (shard || nbytes == 0) && table, "b2_tfrecord_open: NULL argument");
    B2_REQUIRE(max_records >= 1 && max_records <= (1u << 24), "b2_tfrecord_open: max_records out of range");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(table) & 15) == 0, "b2_tfrecord_open: table must be 16-byte aligned");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(shard) & 15) == 0, "b2_tfrecord_open: shard must be 16-byte aligned");
    B2_REQUIRE(nbytes < (1ull << 44), "b2_tfrecord_open: shard too large");
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const TableView v = table_view(table, nbytes, max_records);
    ScanOut o{v.rec_off, v.rec_len, v.hdr, v.tile_start, v.acc, 8};
    scan_kernel<<<1, kScanThreads, 0, s>>>(shard, nbytes, max_records, o, ctx->crc_dev);
    index_kernel<<<(unsigned)((max_records + kIdxWarps - 1) / kIdxWarps), kIdxWarps * 32, 0, s>>>(
        shard, nbytes, v.rec_off, v.rec_len, (int)max_records, v.index, v.hdr, v.tile_start, v.tile2rec);
    ctx->launches += 2;
    B2_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int b2_tfrecord_build(b2_ctx* ctx, const b2_build_desc* descs, int n, uint64_t max_record_bytes,
                                 const uint8_t* scaffold, uint8_t* out, b2_stream stream) {
    B2_REQUIRE(ctx && descs && scaffold && out, "b2_tfrecord_build: NULL argument");
    B2_REQUIRE(n >= 0 && n <= 65535, "b2_tfrecord_build: n must be in [0,65535] per call");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "b2_tfrecord_build: out must be 16-byte aligned");
    if (n == 0) return 0;
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    uint32_t tx = (uint32_t)((max_record_bytes + 15 + kTile - 1) / kTile);
    if (!tx) tx = 1;
    // per-record accumulators live in the context workspace: calls on one context must be stream-ordered
    WsLock ws_lock(ctx);
    if (int e = ws_reserve(ctx, (size_t)n * sizeof(unsigned long long), s)) return e;
    B2_CUDA(cudaMemsetAsync(ctx->ws, 0, (size_t)n * sizeof(unsigned long long), s));
    BuildArgs ba{descs, scaffold, out, ctx->crc_dev, static_cast<unsigned long long*>(ctx->ws)};
    build_kernel<<<dim3((tx + kBuildRun - 1) / kBuildRun, n), kTileThreads, 0, s>>>(ba);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------- host: Example layout
namespace {
void put_varint(std::vector<uint8_t>& v, uint64_t x) {
    while (x >= 0x80) {
        v.push_back((uint8_t)(x | 0x80));
        x >>= 7;
    }
    v.push_back((uint8_t)x);
}
size_t varint_len(uint64_t x) {
    size_t n = 1;
    while (x >= 0x80) { x >>= 7; n++; }
    return n;
}
// entry header for a payload feature: everything up to (not including) the payload bytes
// entry = 0a <elen> [ 0a <klen> key  12 <flen> [ <ftag> <llen> [ 0a <plen> payload ] ] ]
void payload_entry_head(std::vector<uint8_t>& v, const char* key, int kind, uint64_t plen) {
    const size_t klen = strlen(key);
    const uint64_t list_len = plen ? 1 + varint_len(plen) + plen : (kind == 1 ? 2 : 0);
    const uint64_t feat_len = 1 + varint_len(list_len) + list_len;
    const uint64_t entry_len = 1 + varint_len(klen) + klen + 1 + varint_len(feat_len) + feat_len;
    v.push_back(0x0a); put_varint(v, entry_len);
    v.push_back(0x0a); put_varint(v, klen); v.insert(v.end(), key, key + klen);
    v.push_back(0x12); put_varint(v, feat_len);
    v.push_back(kind == 1 ? 0x0a : 0x12); put_varint(v, list_len);
    if (plen || kind == 1) { v.push_back(0x0a); put_varint(v, plen); }
}
uint64_t payload_entry_total(const char* key, int kind, uint64_t plen) {
    std::vector<uint8_t> t;
    payload_entry_head(t, key, kind, plen);
    return t.size() + plen;
}
void int_entry(std::vector<uint8_t>& v, const char* key, int64_t val) {
    const size_t klen = strlen(key);
    const size_t vl = varint_len((uint64_t)val);
    const uint64_t list_len = 1 + 1 + vl, feat_len = 1 + 1 + list_len;
    const uint64_t entry_len = 1 + varint_len(klen) + klen + 1 + 1 + feat_len;
    v.push_back(0x0a); put_varint(v, entry_len);
    v.push_back(0x0a); put_varint(v, klen); v.insert(v.end(), key, key + klen);
    v.push_back(0x12); put_varint(v, feat_len);
    v.push_back(0x1a); put_varint(v, list_len);
    v.push_back(0x0a); put_varint(v, vl); put_varint(v, (uint64_t)val);
}
void bytes_entry(std::vector<uint8_t>& v, const char* key, const uint8_t* data, uint64_t n) {
    payload_entry_head(v, key, 1, n);
    v.insert(v.end(), data, data + n);
}
}  // namespace

extern "C" int b2_example_layout(int kind, uint64_t img_bytes, uint64_t tgt_bytes, int64_t img_h, int64_t img_w,
                                 int64_t img_c, int64_t tgt_h, int64_t tgt_w, const uint8_t* identifier,
                                 uint64_t identifier_len, uint8_t* scaffold, uint64_t cap, uint32_t piece_len[3],
                                 uint64_t* example_len) {
    B2_REQUIRE(kind == 1 || kind == 2, "b2_example_layout: kind must be 1 (BytesList) or 2 (FloatList)");
    B2_REQUIRE(scaffold && piece_len && example_len && (identifier || identifier_len == 0), "b2_example_layout: NULL argument");
    B2_REQUIRE(kind == 1 || ((img_bytes | tgt_bytes) & 3) == 0, "b2_example_layout: FloatList payload must be a multiple of 4 bytes");
    // sorted key order: identifier, image/channels, image/height, image/image_data, image/width,
    //                   target/height, target/target_data, target/width
    std::vector<uint8_t> p0, p1, p2;
    bytes_entry(p0, "identifier", identifier, identifier_len);
    int_entry(p0, "image/channels", img_c);
    int_entry(p0, "image/height", img_h);
    payload_entry_head(p0, "image/image_data", kind, img_bytes);
    int_entry(p1, "image/width", img_w);
    int_entry(p1, "target/height", tgt_h);
    payload_entry_head(p1, "target/target_data", kind, tgt_bytes);
    int_entry(p2, "target/width", tgt_w);
    const uint64_t features_len = p0.size() + img_bytes + p1.size() + tgt_bytes + p2.size();
    std::vector<uint8_t> head;
    head.push_back(0x0a);
    put_varint(head, features_len);
    p0.insert(p0.begin(), head.begin(), head.end());
    B2_REQUIRE(p0.size() + p1.size() + p2.size() <= cap, "b2_example_layout: scaffold buffer too small");
    memcpy(scaffold, p0.data(), p0.size());
    memcpy(scaffold + p0.size(), p1.data(), p1.size());
    memcpy(scaffold + p0.size() + p1.size(), p2.data(), p2.size());
    piece_len[0] = (uint32_t)p0.size();
    piece_len[1] = (uint32_t)p1.size();
    piece_len[2] = (uint32_t)p2.size();
    *example_len = p0.size() + img_bytes + p1.size() + tgt_bytes + p2.size();
    (void)payload_entry_total;
    return 0;
}

/* The scaffolds and descriptor geometry of n records in one call (the per-record form costs the translators one ctypes
 * round trip and a dozen Python objects per chip, which is what bounded them once decode and serialisation ran on the GPU). */
extern "C" int b2_example_layout_batch(int n, const int32_t* kind, const uint64_t* img_bytes, const uint64_t* tgt_bytes,
                                       const int32_t* dims, const uint8_t* ids, const uint64_t* id_off, b2_build_desc* descs,
                                       uint8_t* scaffold, uint64_t scaffold_cap, uint64_t* scaffold_len, uint64_t* total_bytes,
                                       uint64_t* max_record) {
    B2_REQUIRE(n >= 0 && (n == 0 || (kind && img_bytes && tgt_bytes && dims && id_off && descs && scaffold)) && scaffold_len &&
               total_bytes && max_record, "b2_example_layout_batch: NULL argument");
    uint64_t pos = 0, sc = 0, mx = 0;
    for (int i = 0; i < n; i++) {
        const int32_t* d = dims + 5 * (size_t)i;
        uint32_t pl[3];
        uint64_t el = 0;
        B2_REQUIRE(sc + 320 + (id_off[i + 1] - id_off[i]) <= scaffold_cap, "b2_example_layout_batch: scaffold buffer too small");
        if (int e = b2_example_layout(kind[i], img_bytes[i], tgt_bytes[i], d[0], d[1], d[2], d[3], d[4],
                                      ids ? ids + id_off[i] : nullptr, id_off[i + 1] - id_off[i], scaffold + sc,
                                      scaffold_cap - sc, pl, &el)) return e;
        b2_build_desc& o = descs[i];
        o.out_off = pos;
        o.example_len = el;
        o.scaffold_off = sc;
        o.piece_len[0] = pl[0];
        o.piece_len[1] = pl[1];
        o.piece_len[2] = pl[2];
        o.kind = kind[i];
        sc += (uint64_t)pl[0] + pl[1] + pl[2];
        pos += el + 16;
        if (el + 16 > mx) mx = el + 16;
    }
    *scaffold_len = sc;
    *total_bytes = pos;
    *max_record = mx;
    return 0;
}
