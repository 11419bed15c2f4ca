// parse.cu — K2b + K4: the fused per-record pass over an opened TFRecord shard.
//
// Replaces (reference call sites): TFRecordDataset's data-CRC check     parse_tfrecords.ipynb cell 4
//                                   tf.io.parse_single_example / decode_raw / reshape
//                                                                        _tfrecord_image_translation.py:249,306-314,394-407
//                                   cast -> per-band normalise, label -> one-hot (north-star row A17)
//
// Work decomposition.  Record data is cut into 8 KiB tiles on a 16-byte aligned grid anchored at the record's
// (aligned-down) data start.  The kernel is persistent (3 CTAs per SM) and warp-specialised:
//   * the PRODUCER warp draws chunks of q consecutive tiles from a device-side counter, describes each tile in
//     shared memory and starts a TMA bulk copy (cp.async.bulk, SASS UBLKCP) of the tile + 32-byte halo into a ring of
//     shared-memory buffers; an mbarrier per buffer flips when the bytes have landed;
//   * the eight CONSUMER warps compute the tile's CRC-32C contribution from shared memory (the bytes cross HBM
//     exactly once) and run the payload sinks on the same shared-memory tile: raw copy, or uint8 -> (x-mean)/std
//     float32 with 128-bit streaming stores, and label -> one-hot through per-warp shared-memory blocks that are
//     pushed to HBM with TMA bulk stores (cp.async.bulk.global.shared::cta): a label costs ONE 4-byte shared-memory
//     write, the 4*K output bytes per label never pass through registers;
//   * producer and consumers meet only through mbarriers (full / empty per buffer); there is no __syncthreads in
//     the steady state and no second kernel: the CRC state of a thread runs on across the consecutive tiles of a
//     record, the warps of a CTA fold their states through a shared-memory slot when the run of tiles ends, and
//     the last warp there merges { CRC partial, tiles done } into the record's 64-bit accumulator (atomic XOR
//     + atomic add on one address); whoever completes a record un-advances the zero padding, compares with the stored
//     masked CRC and writes the record's status.
//
// CRC-32C without a CRC instruction: the pure CRC (zero init) is linear over GF(2), so
//   * thread i consumes vectors i and i+256 (16 bytes each) of every tile with slice-by-4 table steps; the step
//     after a vector's last word also skips the 4080 bytes to the thread's next vector, in this tile or the next;
//   * when the run ends, one GF(2)[x] multiplication by x^(-128 i) aligns thread i's state with the tile end,
//     the states XOR together, and one more multiplication by a tabulated power of x moves the partial to the
//     end of the record.  The 0xFFFFFFFF init is XORed into the first four data bytes.
#include "tfrecord_common.cuh"

#ifndef B2_WAIT_HINT_NS
#define B2_WAIT_HINT_NS 4000u
#endif
#ifndef B2_STAGES
#define B2_STAGES 2
#endif
#ifndef B2_HOT_BLOCKS
#define B2_HOT_BLOCKS 2
#endif
#ifndef B2_HOT_LABELS
#define B2_HOT_LABELS 64
#endif

namespace b2 {

constexpr int kBufBytes = kTile + 128;   // tile + 32-byte halo, rounded so the second buffer stays 128-byte aligned
constexpr int kHotMaxK = 32;             // one-hot through shared-memory blocks + bulk stores up to this many classes
constexpr int kHotLabels = B2_HOT_LABELS;  // labels per warp block (one or two per lane): one bulk store moves 4*K bytes per label
constexpr int kHotBlocks = B2_HOT_BLOCKS;            // blocks per warp: the bulk store of one overlaps the fill of the other
// Tile buffers in the producer -> consumer ring.  The normalise + one-hot pass is bound by its output traffic and
// short of shared memory (the one-hot blocks), so two do; the CRC-only and raw-copy passes are bound by the CRC chain
// and by how well the bulk loads hide behind it: four buffers (ncu: a third of their stall samples were consumers
// waiting for a tile with two).
// The two normalise + one-hot modes (uint8 BytesList and float32 FloatList payloads) share every resource decision.
__host__ __device__ constexpr bool is_norm(int mode) { return mode == B2_SINK_NORM_ONEHOT || mode == B2_SINK_NORM_ONEHOT_F32; }
// bytes per payload element: 1 for BytesList, 4 for packed FloatList
__host__ __device__ constexpr uint32_t elem_bytes(int mode) { return mode == B2_SINK_NORM_ONEHOT_F32 ? 4u : 1u; }
__host__ __device__ constexpr int stages_for(int mode) { return is_norm(mode) ? B2_STAGES : 4; }
constexpr int kMaxStages = 4;
constexpr int kConsumerWarps = kTileThreads / 32;
constexpr int kCtaThreads = kTileThreads + 32;   // 8 consumer warps + 1 producer warp
constexpr int kRunSlots = 8;             // shared-memory CRC accumulators for runs in flight (> stages)

// ---------------------------------------------------------------- PTX: mbarrier + bulk async copies (TMA, 1-D)
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"     // %2: suspend-time hint (ns): sleep, do not spin
        "@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}" ::"r"(smem_addr(bar)), "r"(parity), "r"(B2_WAIT_HINT_NS) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_addr(dst)),
                 "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_addr(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- arguments
struct ParseArgs {
    const uint8_t* shard;
    uint64_t nbytes;                 // bytes that may be read from shard; ~0 = unknown (never read past a range end)
    const uint64_t* rec_off;
    const uint64_t* rec_len;
    const b2_example_index* index;   // NULL: CRC only
    b2_parse_sink sink;
    const CrcTables* tab;
    // tile -> record map.  Opened shard: tile2rec / tile_start / hdr (device-resident counts).  Otherwise uniform:
    // tile w belongs to record w / tiles_x.
    const uint32_t* tile2rec;
    const uint32_t* tile_start;
    const int64_t* hdr;
    uint32_t tiles_x, n;
    uint32_t q;                      // consecutive tiles per CTA
    unsigned long long* acc;         // per record { CRC partial (low word), tiles accounted for (high word) }: zero on
                                     // entry, zero again on exit
    int32_t* status;                 // per-record status (parse) ...
    uint32_t* crc_out;               // ... or raw CRCs (b2_crc32c)
    int64_t* n_bad;                  // hdr[4] of an opened shard, or NULL
    uint32_t* sched;                 // [0] next chunk of q tiles, [1] CTAs that have finished; both zero between launches
    unsigned long long* prof;        // phase cycle counters (development aid, kProf instantiation only)
    uint32_t row_mask;               // ~0; development probes pass 0 so that every record lands in output row 0 (L2-resident)
};

struct __align__(16) TileJob {
    uint64_t ts, d0, d1;
    uint64_t img_off, img_len, tgt_off, tgt_len;
    uint32_t r, tile, nt, cb, tail, flags;   // flags: 1 valid, 2 sink ok
};

// What the producer knows about the record it is currently cutting into tiles.  Consecutive tiles almost always
// belong to the same record, so the table lookups (tile -> record -> offsets -> feature index: three dependent
// L2 round trips) are paid once per record, not once per tile.
struct RecCache {
    uint32_t r, t0, nt, flags;     // record, its first tile, its tile count, 2 = sinks may run
    uint64_t d0, len;
    uint64_t img_off, img_len, tgt_off, tgt_len;
};

// The sinks' whole verdict on a record, in one place so that rec_lookup (whether they run) and finalize_record (the
// status) cannot disagree.  0: they run.  2: the index refused the record, or it does not fit the normalise + one-hot
// template: both payloads BytesList (NORM_ONEHOT) or packed FloatList (NORM_ONEHOT_F32), the sink's band count, payloads
// as long as the record's dimensions say (else the reference's decode_raw / reshape raises).  3: a payload does not fit
// its output row, or has 2^31 elements or more (the sinks index elements with 32 bits).
template <int kMode>
__device__ __forceinline__ int32_t sink_status(const b2_example_index* ix, const b2_parse_sink& sink) {
    if (ix->status != 0) return 2;
    if (kMode == B2_SINK_RAW) return ix->img_len <= sink.img_stride && ix->tgt_len <= sink.tgt_stride ? 0 : 3;
    constexpr int kKind = kMode == B2_SINK_NORM_ONEHOT_F32 ? 2 : 1;
    constexpr uint64_t kEB = elem_bytes(kMode);
    const int C = sink.channels;
    if (ix->img_kind != kKind || ix->tgt_kind != kKind || ix->channels != C) return 2;
    if (ix->height < 0 || ix->width < 0 || ix->tgt_height < 0 || ix->tgt_width < 0) return 2;
    const uint64_t hw = (uint64_t)ix->height * (uint64_t)ix->width;   // < 2^62; C <= 64 (check_sink)
    const uint64_t thw = (uint64_t)ix->tgt_height * (uint64_t)ix->tgt_width;
    if (hw >= (1ull << 48) || hw * (uint64_t)C * kEB != ix->img_len || thw * kEB != ix->tgt_len) return 2;
    const uint64_t ie = hw * (uint64_t)C, te = thw, K = (uint64_t)sink.num_classes;
    return ie * 4 <= sink.img_stride && te * K * 4 <= sink.tgt_stride && ie < (1ull << 31) && te * K < (1ull << 31) ? 0 : 3;
}

template <int kMode>
__device__ __forceinline__ void rec_lookup(const ParseArgs& a, uint32_t w, RecCache& c) {
    uint32_t r;
    if (a.tile2rec) {
        if (c.r != 0xFFFFFFFFu && w - c.t0 < c.nt) return;               // still inside the cached record
        r = a.tile2rec[w];
        c.t0 = a.tile_start[r];
    } else {
        r = w / a.tiles_x;
        if (r == c.r) return;
        c.t0 = r * a.tiles_x;
    }
    c.r = r;
    c.d0 = a.rec_off[r];
    c.len = a.rec_len[r];
    c.nt = record_tiles(c.d0, c.len);
    c.flags = 0;
    c.img_off = c.img_len = c.tgt_off = c.tgt_len = 0;
    if (kMode != B2_SINK_NONE && a.index != nullptr) {
        const b2_example_index* ix = a.index + r;
        if (sink_status<kMode>(ix, a.sink) == 0) {
            c.flags = 2;
            c.img_off = ix->img_off;
            c.img_len = ix->img_len;
            c.tgt_off = ix->tgt_off;
            c.tgt_len = ix->tgt_len;
        }
    }
}

// producer: describe tile w and start its copy into buf
template <int kMode>
__device__ __forceinline__ void make_job(const ParseArgs& a, uint32_t w, RecCache& c, TileJob* j, uint8_t* buf, uint64_t* bar) {
    rec_lookup<kMode>(a, w, c);
    const uint32_t r = c.r, tile = w - c.t0, nt = c.nt;
    const uint64_t d0 = c.d0, len = c.len;
    j->r = r;
    j->tile = tile;
    j->nt = nt;
    if (tile >= nt) {   // uniform map only: this record has fewer tiles than the longest one
        j->flags = 0;
        mbar_arrive(bar);
        return;
    }
    const uint64_t d1 = d0 + len, ts = (d0 & ~15ull) + (uint64_t)tile * kTile, te = ts + kTile;
    j->ts = ts;
    j->d0 = d0;
    j->d1 = d1;
    j->img_off = c.img_off;
    j->img_len = c.img_len;
    j->tgt_off = c.tgt_off;
    j->tgt_len = c.tgt_len;
    j->flags = 1 | c.flags;
    // bytes to stage: [ts, min(te + 32, d1)), never touching shard[lim...]
    const uint64_t lim = a.nbytes != ~0ull ? a.nbytes : d1;
    uint64_t want = (d1 + 15) & ~15ull;
    if (want > te + 32) want = te + 32;
    uint32_t cb, tail = 0;
    if (len == 0) {
        cb = 0;
    } else if (want <= lim) {
        cb = (uint32_t)(want - ts);
    } else {
        cb = (uint32_t)((lim - ts) & ~15ull);
        const uint64_t end = d1 < lim ? d1 : lim;
        tail = end > ts + cb ? (uint32_t)(end - ts - cb) : 0;
    }
    j->cb = cb;
    j->tail = tail;
    for (uint32_t i = 0; i < tail; i++) buf[cb + i] = a.shard[ts + cb + i];   // < 16 bytes, last tile of a shard only
    if (cb) {
        mbar_expect_tx(bar, cb);          // release: the job and the tail bytes are visible to whoever sees the phase flip
        bulk_g2s(buf, a.shard + ts, cb, bar);
    } else {
        mbar_arrive(bar);
    }
}

// whether tile [ts, te) holds any byte of payload [po, po + len) (absolute)
__device__ __forceinline__ bool tile_holds(uint64_t ts, uint64_t te, uint64_t po, uint64_t len) {
    return len != 0 && po < te && po + len > ts;
}

// raw byte copy of payload range [po, po+pl) (absolute) into dst, for the part owned by tile [ts, te)
__device__ __forceinline__ void sink_raw(const uint32_t* buf32, const uint8_t* buf8, uint64_t ts, uint64_t te,
                                         uint64_t po, uint64_t pl, uint8_t* dst) {
    if (!tile_holds(ts, te, po, pl)) return;
    const bool al = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
    const uint64_t lo = po > ts ? po : ts, hi = (po + pl < te) ? po + pl : te;  // absolute bytes in this tile
    if (al) {
        // 16-byte destination groups whose FIRST byte lies in the tile; last partial group done bytewise
        const uint64_t g_lo = (lo - po + 15) >> 4, g_hi = (hi - po + 15) >> 4;
        const uint64_t full = pl >> 4;
        for (uint64_t g = g_lo + threadIdx.x; g < g_hi; g += kTileThreads) {
            const uint32_t o = (uint32_t)(po + 16 * g - ts);
            if (g < full) {
                uint4 v;
                v.x = smem_u32_unaligned(buf32, o);
                v.y = smem_u32_unaligned(buf32, o + 4);
                v.z = smem_u32_unaligned(buf32, o + 8);
                v.w = smem_u32_unaligned(buf32, o + 12);
                st_cs(reinterpret_cast<uint4*>(dst + 16 * g), v);
            } else {
                for (uint64_t b = 16 * g; b < pl; b++) dst[b] = buf8[o + (b - 16 * g)];
            }
        }
    } else {
        for (uint64_t p = lo + threadIdx.x; p < hi; p += kTileThreads) dst[p - po] = buf8[p - ts];
    }
}

// (x - mean) / std, bit-identical with IEEE division.  Fast path: q = d * r, corrected by one residual step
// (r = correctly rounded 1/std): 3 FP32 instructions instead of the ~10 of a full division.  Whether the fast path
// reproduces the division for EVERY byte value of EVERY band is checked once per CTA (256*C cases); if any case
// differs (or std is 0 / non-finite) the whole launch uses the division.
__device__ __forceinline__ float norm_fast(float d, float sd, float rc) {
    const float q = __fmul_rn(d, rc);
    const float rem = __fmaf_rn(-q, sd, d);
    return __fmaf_rn(rem, rc, q);
}

// The sinks below write the part of payload [po, po + len) (absolute bytes; elements of kEB bytes: uint8 or little-endian
// float32) that tile [ts, te) owns.  Callers check tile_holds before computing the output row (keeps registers down).
// base = po - ts: the payload start in the tile buffer (wraps when po < ts; base + kEB * element is in [0, kTile) mod 2^32).

// float4 group g of an output row of n floats (full4 = n / 4 whole groups): one streaming store, or the last 1..3 floats
__device__ __forceinline__ void store_group(float* dst, uint32_t g, uint32_t full4, uint32_t n, const float (&f)[4]) {
    if (g < full4) st_cs(reinterpret_cast<float4*>(dst) + g, make_float4(f[0], f[1], f[2], f[3]));
    else for (uint32_t k = 0; k < 3; k++) if (4 * g + k < n) dst[4 * g + k] = f[k];
}

// label l's class (-1: all-zero row)
template <uint32_t kEB>
__device__ __forceinline__ int payload_class(const uint8_t* buf8, const uint32_t* buf32, uint32_t base, uint32_t l, int K) {
    if constexpr (kEB == 1) return label_class<uint8_t>(buf8[base + l], K);
    else return label_class<float>(__uint_as_float(smem_u32_unaligned(buf32, base + 4 * l)), K);
}

// image -> (x - mean) / std float32; thread tid < S takes float4 groups tid, tid + S, ... (S: img_S in the kernel)
template <uint32_t kEB>
__device__ __forceinline__ void sink_image(const uint32_t* buf32, uint64_t ts, uint64_t te, uint64_t po, uint64_t len,
                                           float* dst, uint32_t S, const float* s_mean, const float* s_std,
                                           const float* s_rcp, int C, bool exact_div) {
    const uint32_t pl = (uint32_t)(len / kEB);   // elements
    const uint64_t lo = po > ts ? po : ts, hi = (po + (uint64_t)pl * kEB < te) ? po + (uint64_t)pl * kEB : te;
    // float4 group g = image elements [4g, 4g+4) = payload bytes [4 kEB g, 4 kEB (g+1)); owned by the tile that holds its
    // first byte, its last bytes may sit in the halo
    const uint32_t g_lo = (uint32_t)((lo - po + 4 * kEB - 1) / (4 * kEB)), g_hi = (uint32_t)((hi - po + 4 * kEB - 1) / (4 * kEB)),
                   full4 = pl >> 2;
    const uint32_t base = (uint32_t)(po - ts);
    uint32_t g = g_lo + threadIdx.x;
    float mu[4], sd[4], rc[4];
    {
        uint32_t ch = (4u * g) % (uint32_t)C;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            mu[k] = s_mean[ch];
            sd[k] = s_std[ch];
            rc[k] = s_rcp[ch];
            ch = (ch + 1 == (uint32_t)C) ? 0 : ch + 1;
        }
    }
    for (; g < g_hi; g += S) {
        float f[4];
        if constexpr (kEB == 1) {
            const uint32_t x = smem_u32_unaligned(buf32, base + 4 * g);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                // byte k -> float, exactly: 0x4B000000 | v is 2^23 + v
                const float v = __uint_as_float(__byte_perm(x, 0x4B000000u, 0x7540 + k)) - 8388608.0f;
                const float d = __fsub_rn(v, mu[k]);
                f[k] = exact_div ? __fdiv_rn(d, sd[k]) : norm_fast(d, sd[k], rc[k]);
            }
        } else {
            // FloatList payloads start at any byte residue: four funnel-shifted words
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float v = __uint_as_float(smem_u32_unaligned(buf32, base + 16 * g + 4 * k));
                f[k] = __fdiv_rn(__fsub_rn(v, mu[k]), sd[k]);
            }
        }
        store_group(dst, g, full4, pl, f);
    }
}

// A consumer warp's kHotBlocks one-hot blocks of kHotLabels*K floats + 4 (float kHotLabels*K is a dummy, never stored)
struct HotBlocks {
    float* blk;                     // this warp's first block
    uint32_t a0, a1, b0, b1;        // the floats this lane set last time in block 0 / block 1
    uint32_t it;                    // blocks filled so far
};

// label -> one-hot float32, K <= kHotMaxK.  A warp's blocks are zero but for ONE 1.0f per label (a label costs one 4-byte
// shared-memory write) and go to HBM with one TMA bulk store each; labels without a class write the dummy, so nothing is
// predicated.  Work unit = 4 labels (4K floats: whole 16-byte groups, 16-byte aligned in the output), owned by the tile
// holding its first label; later labels may sit in the halo.
template <uint32_t kEB>
__device__ __forceinline__ void sink_onehot_smem(const uint8_t* buf8, const uint32_t* buf32, uint64_t ts, uint64_t te,
                                                 uint64_t po, uint64_t len, float* dst, int K, HotBlocks& h) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t pl = (uint32_t)(len / kEB);   // labels
    const uint64_t lo = po > ts ? po : ts, hi = (po + (uint64_t)pl * kEB < te) ? po + (uint64_t)pl * kEB : te;
    const uint32_t base = (uint32_t)(po - ts);
    const uint32_t dummy = kHotLabels * K;
    const uint32_t j_lo = (uint32_t)((lo - po + 4 * kEB - 1) / (4 * kEB)), j_hi = (uint32_t)((hi - po + 4 * kEB - 1) / (4 * kEB));
    const uint32_t L_beg = 4 * j_lo, L_end = (4 * j_hi < pl) ? 4 * j_hi : pl;
    for (uint32_t L0 = L_beg + warp * kHotLabels; L0 < L_end; L0 += kConsumerWarps * kHotLabels) {
        const uint32_t hb = kHotBlocks > 1 ? (h.it & 1) : 0;
        h.it++;
        float* hot = h.blk + hb * (kHotLabels * K + 4);
        if (lane == 0) bulk_wait_read<kHotBlocks - 1>();   // the store that last used this block has read it
        __syncwarp();
        hot[hb ? h.b0 : h.a0] = 0.0f;
        hot[hb ? h.b1 : h.a1] = 0.0f;
        constexpr uint32_t kPerLane = kHotLabels / 32;
        const uint32_t l0 = L0 + kPerLane * lane;
        uint32_t slot0 = dummy, slot1 = dummy;
        if (l0 < L_end) {
            const int k = payload_class<kEB>(buf8, buf32, base, l0, K);
            if (k >= 0) slot0 = (kPerLane * lane) * K + k;
        }
        if (kPerLane > 1 && l0 + 1 < L_end) {
            const int k = payload_class<kEB>(buf8, buf32, base, l0 + 1, K);
            if (k >= 0) slot1 = (kPerLane * lane + 1) * K + k;
        }
        hot[slot0] = 1.0f;
        hot[slot1] = 1.0f;
        if (hb) { h.b0 = slot0; h.b1 = slot1; } else { h.a0 = slot0; h.a1 = slot1; }
        fence_proxy_async();
        __syncwarp();
        const uint32_t nl = (L_end - L0 < (uint32_t)kHotLabels) ? L_end - L0 : (uint32_t)kHotLabels;
        const uint32_t nfl = nl * K, nb16 = (nfl * 4) & ~15u;
        if (lane == 0) {
            if (nb16) bulk_s2g(dst + (size_t)L0 * K, hot, nb16);
            bulk_commit();
        }
        if ((uint32_t)lane < (nfl & 3)) dst[(size_t)L0 * K + (nfl & ~3u) + lane] = hot[(nfl & ~3u) + lane];
    }
}

// label -> one-hot float32 for any K (used above kHotMaxK): float4 group g holds one-hot floats [4g, 4g+4), owned by the
// tile of label 4g/K
template <uint32_t kEB>
__device__ __forceinline__ void sink_onehot_generic(const uint8_t* buf8, const uint32_t* buf32, uint64_t ts, uint64_t te,
                                                    uint64_t po, uint64_t len, float* dst, int K) {
    const uint32_t pl = (uint32_t)(len / kEB);   // labels
    const uint64_t lo = po > ts ? po : ts, hi = (po + (uint64_t)pl * kEB < te) ? po + (uint64_t)pl * kEB : te;
    const uint32_t base = (uint32_t)(po - ts);
    const uint32_t nfl = pl * (uint32_t)K;
    const uint32_t g_lo = (uint32_t)(((lo - po + kEB - 1) / kEB * K + 3) >> 2),
                   g_hi = (uint32_t)(((hi - po + kEB - 1) / kEB * K + 3) >> 2), full4 = nfl >> 2;
    for (uint32_t g = g_lo + threadIdx.x; g < g_hi; g += kTileThreads) {
        const uint32_t f0 = 4 * g;
        uint32_t l = f0 / (uint32_t)K;
        uint32_t cc = f0 - l * (uint32_t)K;
        float f[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            // a label without a class reads as 0xFFFFFFFF, which equals no class index
            const uint32_t lab = (l < pl) ? (uint32_t)payload_class<kEB>(buf8, buf32, base, l, K) : 0xFFFFFFFFu;
            f[k] = (lab == cc) ? 1.0f : 0.0f;
            if (++cc == (uint32_t)K) {
                cc = 0;
                l++;
            }
        }
        store_group(dst, g, full4, nfl, f);
    }
}

struct RecRef {   // what finalize_record needs to know about the record
    uint32_t r, nt;
    uint64_t d0, d1;
};

template <int kMode>
__device__ inline void finalize_record(const ParseArgs& a, const RecRef& j, uint32_t acc) {
    const uint32_t r = j.r;
    const uint64_t d0 = j.d0, len = j.d1 - j.d0;
    const bool want_crc = a.sink.verify_crc || a.crc_out;
    uint32_t crc = 0;
    if (want_crc) {
        if (len < 4) {   // the init XOR does not fit in the message: bytewise
            uint32_t s = 0xFFFFFFFFu;
            for (uint64_t i = 0; i < len; i++) s = (s >> 8) ^ __ldg(&a.tab->t4[3][(s ^ a.shard[d0 + i]) & 0xff]);
            crc = ~s;
        } else {
            // acc sits at the end of the last tile; un-advance by the zero padding after the record end
            const uint64_t pad = (d0 & ~15ull) + (uint64_t)j.nt * kTile - j.d1;
            acc = multmodp(__ldg(&a.tab->xinv16[pad >> 4]), acc);
            acc = multmodp(__ldg(&a.tab->xinvb[pad & 15]), acc);
            crc = ~acc;
        }
    }
    if (a.crc_out) {
        a.crc_out[r] = crc;
        return;
    }
    int32_t st = 0;
    if (a.sink.verify_crc) {
        uint32_t stored = ~mask_crc(crc);
        if (a.nbytes == ~0ull || j.d1 + 4 <= a.nbytes) {
            stored = 0;
            for (int k = 0; k < 4; k++) stored |= (uint32_t)a.shard[j.d1 + k] << (8 * k);
        }
        if (stored != mask_crc(crc)) st = 1;
    }
    if (kMode != B2_SINK_NONE && st == 0 && a.index) st = sink_status<kMode>(a.index + r, a.sink);
    a.status[r] = st;
    if (st != 0 && a.n_bad) atomicAdd(reinterpret_cast<unsigned long long*>(a.n_bad), 1ull);
}

__device__ __forceinline__ uint32_t crc_tile_step(uint32_t s, const uint4* buf4, const CrcSmem* cs, const TileJob& j,
                                                  bool interior) {
    return crc_running_step(s, buf4, cs, j.ts, j.d0, j.d1, j.tile == 0, interior);
}

struct Run {             // consecutive tiles of one record handled by this CTA (uniform across the consumer warps)
    uint32_t r, nt, last_tile, tiles;
    uint64_t d0, d1;
    bool open;
};
struct RunAcc {          // shared-memory meeting point of the eight consumer warps at the end of a run
    uint32_t crc, warps;
};

// Close a run.  No CTA-wide barrier: every consumer warp folds its lanes' CRC states, XORs the result into the run's
// shared-memory slot and counts itself; the warp that arrives last moves the partial to the end of the record and
// merges { CRC, tiles } into the record's 64-bit accumulator with an atomic XOR and an atomic add on the same address
// (applied in program order, so no fences are needed), finalising the record when its tile count is complete.  The other warps are already working
// on the next tile.  Every warp flushes a run in the same loop iteration `it`, at most one run per iteration, and its
// slot is `it` mod kRunSlots: a slot comes round again kRunSlots iterations later, and no warp can be more than kStages
// (< kRunSlots) iterations ahead of the slowest, whose arrival on the buffer's empty barrier the producer waits for.
template <int kMode>
__device__ __forceinline__ void run_flush(const ParseArgs& a, Run& run, uint32_t& s, uint32_t it, bool want_crc,
                                          RunAcc* racc) {
    const int tid = threadIdx.x, lane = tid & 31;
    RunAcc* ra = racc + (it & (kRunSlots - 1));
    const bool crc = want_crc && run.d1 - run.d0 >= 4;
    if (crc) {
        uint32_t t = multmodp_fast(__ldg(&a.tab->xinv16[tid]), s);
#pragma unroll
        for (int o = 16; o; o >>= 1) t ^= __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0 && t) atomicXor(&ra->crc, t);
    }
    if (lane == 0) {
        __threadfence_block();
        if (atomicAdd(&ra->warps, 1u) == kConsumerWarps - 1) {
            __threadfence_block();
            uint32_t c = atomicExch(&ra->crc, 0u);
            ra->warps = 0;
            if (crc) c = multmodp_fast(tile_power(a.tab, run.nt - 1 - run.last_tile), c);
            // XOR into the low word, then count in the high word: two atomics on ONE address are applied in program
            // order, so whoever sees the count complete also sees every partial (no fence, no retry loop)
            unsigned long long* acc = a.acc + run.r;
            if (c) atomicXor(acc, (unsigned long long)c);
            const unsigned long long upd = atomicAdd(acc, (unsigned long long)run.tiles << 32) + ((unsigned long long)run.tiles << 32);
            if ((uint32_t)(upd >> 32) == run.nt) {
                *acc = 0ull;               // re-arm for the next launch; nobody else touches a finished record
                RecRef rr{run.r, run.nt, run.d0, run.d1};
                finalize_record<kMode>(a, rr, (uint32_t)upd);
            }
        }
    }
    s = 0;
    run.open = false;
}

// Development aid: cycles spent by lane 0 of every consumer warp in each phase of the tile loop (B2_PARSE_PROFILE=1).
#define PROF_BEGIN() \
    long long prof_t = 0; \
    unsigned long long prof_acc[7] = {0, 0, 0, 0, 0, 0, 0}; \
    if (kProf && lane == 0) prof_t = clock64();
#define PROF_MARK(k) \
    if (kProf && lane == 0) { \
        const long long t_ = clock64(); \
        prof_acc[k] += (unsigned long long)(t_ - prof_t); \
        prof_t = t_; \
    }
#define PROF_END() \
    if (kProf && lane == 0) { \
        for (int k_ = 0; k_ < 7; k_++) atomicAdd(&a.prof[k_ + (warp == 0 ? 0 : 8)], prof_acc[k_]); \
    }

// Warp-specialised persistent kernel: warp 8 is the PRODUCER (draws chunks of q tiles from the device-side counter,
// describes each tile in shared memory and starts its TMA bulk copy into a ring of kStages buffers), warps 0..7 are
// CONSUMERS (CRC, payload sinks).  They meet only through mbarriers: full[s] flips when tile s has landed, empty[s]
// when all eight consumer warps are done with it — there is no __syncthreads in the steady state.
template <int kMode, bool kProf = false>
__global__ void __launch_bounds__(kCtaThreads, is_norm(kMode) ? 3 : 5)
fused_parse_kernel(const ParseArgs a) {
    constexpr int kStages = stages_for(kMode);
    static_assert(kStages <= kMaxStages && kRunSlots > kStages, "ring sizes");
    extern __shared__ __align__(128) uint8_t dyn[];
    __shared__ CrcSmem cs;
    __shared__ TileJob job[kStages];
    __shared__ __align__(8) uint64_t full[kStages], empty[kStages];
    __shared__ RunAcc racc[kRunSlots];
    __shared__ float s_mean[64], s_std[64], s_rcp[64];
    __shared__ int s_exact_div;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const uint64_t total = a.hdr ? (uint64_t)a.hdr[2] : (uint64_t)a.n * a.tiles_x;
    const bool want_crc = a.sink.verify_crc || a.crc_out;
    const int C = a.sink.channels, K = a.sink.num_classes;
    const bool use_hot = K <= kHotMaxK;
    float* hot_all = reinterpret_cast<float*>(dyn + kStages * kBufBytes);

    if (want_crc) load_crc_tables(&cs, a.tab);
    if (is_norm(kMode)) {
        if (tid == 0) s_exact_div = 0;
        for (int c = tid; c < C; c += kCtaThreads) {
            s_mean[c] = a.sink.mean[c];
            s_std[c] = a.sink.std[c];
            s_rcp[c] = __frcp_rn(a.sink.std[c]);
        }
        if (use_hot)
            for (int i = tid; i < kConsumerWarps * kHotBlocks * (kHotLabels * K + 4); i += kCtaThreads) hot_all[i] = 0.0f;
    }
    if (tid == 0) {
        for (int k = 0; k < kStages; k++) {
            mbar_init(&full[k], 1);
            mbar_init(&empty[k], kConsumerWarps);
        }
        for (int k = 0; k < kRunSlots; k++) racc[k].crc = racc[k].warps = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (kMode == B2_SINK_NORM_ONEHOT) {   // NORM_ONEHOT_F32 always divides: float inputs have no finite set to check
        int bad = 0;
        for (int i = tid; i < C * 256; i += kCtaThreads) {
            const int c = i >> 8;
            const float d = __fsub_rn((float)(i & 255), s_mean[c]);
            bad |= __float_as_uint(norm_fast(d, s_std[c], s_rcp[c])) != __float_as_uint(__fdiv_rn(d, s_std[c]));
        }
        if (bad) s_exact_div = 1;
        __syncthreads();
    }

    if (warp == kConsumerWarps) {
        // ------------------------------------------------------------------------------------------ producer
        if (lane != 0) return;
        uint32_t feed_w = 0, feed_left = 0;
        RecCache rc;
        rc.r = 0xFFFFFFFFu;
        rc.t0 = rc.nt = 0;
        for (uint32_t it = 0;; it++) {
            const uint32_t slot = it % kStages, use = it / kStages;
            if (use > 0) mbar_wait(&empty[slot], (use - 1) & 1);
            if (feed_left == 0) {
                const uint64_t w = (uint64_t)atomicAdd(&a.sched[0], 1u) * a.q;
                if (w >= total) {
                    job[slot].flags = 4;
                    mbar_arrive(&full[slot]);
                    break;
                }
                feed_w = (uint32_t)w;
                feed_left = (uint32_t)(total - w < a.q ? total - w : a.q);
            }
            make_job<kMode>(a, feed_w, rc, &job[slot], dyn + slot * kBufBytes, &full[slot]);
            feed_w++;
            feed_left--;
        }
        // the last CTA out re-arms the chunk counter for the next launch
        __threadfence();
        if (atomicAdd(&a.sched[1], 1u) == gridDim.x - 1) {
            a.sched[0] = 0;
            a.sched[1] = 0;
        }
        return;
    }

    // ---------------------------------------------------------------------------------------------- consumers
    const bool exact_div = kMode == B2_SINK_NORM_ONEHOT && s_exact_div != 0;
    // image loop stride: the largest S <= 256 with 4 S a multiple of C, so that a thread's four bytes always fall on
    // the same four bands and their constants stay in registers
    uint32_t img_S = kTileThreads;
    if (is_norm(kMode)) {
        const uint32_t m = (C % 4 == 0) ? C / 4 : ((C % 2 == 0) ? C / 2 : C);
        img_S = kTileThreads - (kTileThreads % m);
    }
    uint32_t s = 0;                       // running CRC state of this thread
    Run run;
    run.open = false;
    const uint32_t hot_dummy = kHotLabels * K;
    HotBlocks hot{hot_all + warp * kHotBlocks * (kHotLabels * K + 4), hot_dummy, hot_dummy, hot_dummy, hot_dummy, 0};
    PROF_BEGIN();

    for (uint32_t it = 0;; it++) {
        const uint32_t slot = it % kStages, use = it / kStages;
        mbar_wait(&full[slot], use & 1);
        PROF_MARK(0);
        const TileJob& j = job[slot];
        const uint32_t flags = j.flags;
        const bool valid = (flags & 1) != 0;
        if (run.open && (!valid || j.r != run.r || j.tile != run.last_tile + 1)) run_flush<kMode>(a, run, s, it, want_crc, racc);
        PROF_MARK(5);
        if (flags & 4) break;
        if (valid) {
            const uint8_t* buf8 = dyn + slot * kBufBytes;
            const uint4* buf4 = reinterpret_cast<const uint4*>(buf8);
            const uint32_t* buf32 = reinterpret_cast<const uint32_t*>(buf8);
            const uint64_t ts = j.ts, te = ts + kTile;
            const uint64_t d0 = j.d0, d1 = j.d1;
            if (!run.open) {
                run.open = true;
                run.r = j.r;
                run.nt = j.nt;
                run.d0 = d0;
                run.d1 = d1;
                run.tiles = 0;
            }
            run.tiles++;
            run.last_tile = j.tile;
            if (want_crc && d1 - d0 >= 4) s = crc_tile_step(s, buf4, &cs, j, j.tile != 0 && te <= d1);
            PROF_MARK(1);
            if (kMode == B2_SINK_RAW && (flags & 2)) {
                if (a.sink.img_out)
                    sink_raw(buf32, buf8, ts, te, j.img_off, j.img_len, static_cast<uint8_t*>(a.sink.img_out) + (uint64_t)(j.r & a.row_mask) * a.sink.img_stride);
                if (a.sink.tgt_out)
                    sink_raw(buf32, buf8, ts, te, j.tgt_off, j.tgt_len, static_cast<uint8_t*>(a.sink.tgt_out) + (uint64_t)(j.r & a.row_mask) * a.sink.tgt_stride);
            }
            if (is_norm(kMode) && (flags & 2)) {
                constexpr uint32_t kEB = elem_bytes(kMode);
                if (a.sink.img_out && (uint32_t)tid < img_S && tile_holds(ts, te, j.img_off, j.img_len))
                    sink_image<kEB>(buf32, ts, te, j.img_off, j.img_len,
                                    reinterpret_cast<float*>(static_cast<uint8_t*>(a.sink.img_out) + (uint64_t)(j.r & a.row_mask) * a.sink.img_stride),
                                    img_S, s_mean, s_std, s_rcp, C, exact_div);
                PROF_MARK(2);
                if (a.sink.tgt_out && tile_holds(ts, te, j.tgt_off, j.tgt_len)) {
                    float* dst = reinterpret_cast<float*>(static_cast<uint8_t*>(a.sink.tgt_out) + (uint64_t)(j.r & a.row_mask) * a.sink.tgt_stride);
                    if (use_hot) sink_onehot_smem<kEB>(buf8, buf32, ts, te, j.tgt_off, j.tgt_len, dst, K, hot);
                    else sink_onehot_generic<kEB>(buf8, buf32, ts, te, j.tgt_off, j.tgt_len, dst, K);
                }
                PROF_MARK(3);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[slot]);   // this warp is done with the buffer and its job
        PROF_MARK(4);
    }
    if (is_norm(kMode) && lane == 0) bulk_wait_read<0>();   // shared memory must outlive the bulk stores
    PROF_END();
}

}  // namespace b2

using namespace b2;

namespace {

bool g_smem_ready[64];   // per device: the kernels' shared-memory opt-ins are set

constexpr size_t dyn_bytes(int mode, int K) {
    return (size_t)stages_for(mode) * kBufBytes +
           (is_norm(mode) && K <= kHotMaxK ? (size_t)(kTileThreads / 32) * kHotBlocks * (kHotLabels * K + 4) * sizeof(float) : 0);
}
// The one-hot blocks at K = kHotMaxK need 145 KiB; the kernel's static shared memory (~9 KiB, ptxas -v) comes on top, and
// both must fit the 227 KiB a block may opt into on sm_100.
constexpr size_t kNormDynMax = dyn_bytes(B2_SINK_NORM_ONEHOT, kHotMaxK);

// Raise a kernel's dynamic shared-memory ceiling to dyn after checking that static + dyn fits the device's per-block limit.
template <typename F>
int set_dyn_smem(F* kernel, size_t dyn, int device) {
    cudaFuncAttributes fa;
    B2_CUDA(cudaFuncGetAttributes(&fa, kernel));
    int optin = 0;
    B2_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    B2_REQUIRE(fa.sharedSizeBytes + dyn <= (size_t)optin, "fused parse: shared memory of the largest launch exceeds the per-block limit");
    B2_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    return 0;
}

// The kernel that runs a sink mode; prof picks the NORM_ONEHOT instantiation with the per-phase cycle counters.
using ParseKernel = void (*)(const ParseArgs);
ParseKernel fused_kernel(int mode, bool prof) {
    const ParseKernel k[] = {fused_parse_kernel<B2_SINK_NONE>, fused_parse_kernel<B2_SINK_RAW>, fused_parse_kernel<B2_SINK_NORM_ONEHOT>,
                             fused_parse_kernel<B2_SINK_NORM_ONEHOT_F32>};
    if (mode == B2_SINK_NORM_ONEHOT && prof) return fused_parse_kernel<B2_SINK_NORM_ONEHOT, true>;
    return mode >= B2_SINK_NONE && mode <= B2_SINK_NORM_ONEHOT_F32 ? k[mode] : nullptr;
}

int launch_fused(b2_ctx* ctx, const ParseArgs& pa, uint64_t max_tiles, cudaStream_t s) {
    if (!g_smem_ready[ctx->device & 63]) {
        // opt-in ceilings of every kernel; the normalise + one-hot modes: what their largest launch (K = kHotMaxK) asks
        // for.  A ceiling only: occupancy follows each launch's actual request.
        for (int mode = B2_SINK_NONE; mode <= B2_SINK_NORM_ONEHOT_F32; mode++)
            for (int prof = 0; prof <= (mode == B2_SINK_NORM_ONEHOT); prof++)   // only NORM_ONEHOT has a profiling twin
                if (int e = set_dyn_smem(fused_kernel(mode, prof), is_norm(mode) ? kNormDynMax : 96 * 1024, ctx->device)) return e;
        g_smem_ready[ctx->device & 63] = true;
    }
    const ParseKernel kernel = fused_kernel(pa.sink.mode, pa.prof != nullptr);
    B2_REQUIRE(kernel, "fused parse: no kernel for this sink mode");
    // persistent grid: as many CTAs as fit on the GPU at once (4 per SM), never more than there are chunks
    const uint64_t chunks = (max_tiles + pa.q - 1) / pa.q;
    const uint64_t resident = (uint64_t)ctx->sm_count * (is_norm(pa.sink.mode) ? 3 : 5);
    const unsigned grid = (unsigned)(chunks < resident ? chunks : resident);
    kernel<<<grid, kCtaThreads, dyn_bytes(pa.sink.mode, pa.sink.num_classes), s>>>(pa);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

int check_sink(const b2_parse_sink* sink, const char* who) {
    if (is_norm(sink->mode)) {
        const std::string m = sink->mode == B2_SINK_NORM_ONEHOT ? ": NORM_ONEHOT" : ": NORM_ONEHOT_F32";
        B2_REQUIRE(sink->mean && sink->std && sink->channels >= 1 && sink->channels <= 64 && sink->num_classes >= 1,
                   std::string(who) + m + " needs mean/std, 1..64 channels and num_classes >= 1");
        B2_REQUIRE((reinterpret_cast<uintptr_t>(sink->img_out) & 15) == 0 && (sink->img_stride & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(sink->tgt_out) & 15) == 0 && (sink->tgt_stride & 15) == 0,
                   std::string(who) + m + " outputs and strides must be 16-byte aligned");
    } else {
        B2_REQUIRE(sink->mode == B2_SINK_NONE || sink->mode == B2_SINK_RAW, std::string(who) + ": unknown sink mode");
    }
    return 0;
}

// Development builds (-DB2_DEV_KNOBS) can alias every output row onto row 0 to time the kernel without its
// output footprint (the roofline experiment in DESIGN.md).  The shipped library has no such switch.
uint32_t dev_row_mask() {
#ifdef B2_DEV_KNOBS
    return getenv("B2_DEBUG_ROW0") ? 0u : ~0u;
#else
    return ~0u;
#endif
}

// Tiles per scheduler chunk (= the longest run whose per-thread CRC state is carried): 2 keeps the output streams of the
// uint8 normalise + one-hot pass balanced; the CRC-only, raw and float32 normalise + one-hot passes amortise the per-run
// alignment multiply over 8 (NORM_ONEHOT_F32 reads 4 bytes per output float and is CRC-bound: cfg3 records with CRC
// take 6.2 us at q = 2, 5.5 us at 4, 5.4 us at 8 on a B200 at 1000 W).
uint32_t tiles_per_cta(int mode) {
#ifdef B2_DEV_KNOBS
    static int q = -1;
    if (q < 0) {
        const char* e = getenv("B2_PARSE_TILES_PER_CTA");
        q = e ? atoi(e) : 0;
        if (q < 0) q = 0;
        if (q > 64) q = 64;
    }
    if (q) return (uint32_t)q;
#endif
    return mode == B2_SINK_NORM_ONEHOT ? 2u : 8u;
}

// Per-phase cycle counters are a development-build feature; the shipped library never reads the environment per call.
unsigned long long* dev_profile(b2_ctx* ctx) {
#ifdef B2_DEV_KNOBS
    return getenv("B2_PARSE_PROFILE") ? ctx->prof_dev : nullptr;
#else
    (void)ctx;
    return nullptr;
#endif
}

// A launch's arguments: the fields every launch sets; the rest start zeroed.
ParseArgs parse_args(b2_ctx* ctx, const uint8_t* shard, uint64_t nbytes, const uint64_t* rec_off, const uint64_t* rec_len,
                     const b2_example_index* index, const b2_parse_sink& sink, int32_t* status) {
    ParseArgs pa{};
    pa.shard = shard;
    pa.nbytes = nbytes;
    pa.rec_off = rec_off;
    pa.rec_len = rec_len;
    pa.index = index;
    pa.sink = sink;
    pa.tab = ctx->crc_dev;
    pa.q = tiles_per_cta(sink.mode);
    pa.status = status;
    pa.row_mask = ~0u;
    return pa;
}

// Uniform tile map for n records of at most max_len bytes: tile w belongs to record w / tiles_x.  The per-record
// accumulators and the scheduler words live in the context workspace: calls on one context must be stream-ordered.
int launch_uniform(b2_ctx* ctx, ParseArgs& pa, int n, uint64_t max_len, cudaStream_t s, const char* who) {
    uint64_t tx = (max_len + 15 + kTile - 1) / kTile;
    if (!tx) tx = 1;
    B2_REQUIRE(tx * (uint64_t)n < (1ull << 32), std::string(who) + ": too many tiles for one call");
    WsLock ws_lock(ctx);
    if (int e = ws_reserve(ctx, (size_t)n * 8 + 8, s)) return e;
    B2_CUDA(cudaMemsetAsync(ctx->ws, 0, (size_t)n * 8 + 8, s));
    pa.tiles_x = (uint32_t)tx;
    pa.n = (uint32_t)n;
    pa.acc = static_cast<unsigned long long*>(ctx->ws);             // n per-record accumulators ...
    pa.sched = reinterpret_cast<uint32_t*>(pa.acc + n);              // ... then the scheduler's two words
    return launch_fused(ctx, pa, tx * (uint64_t)n, s);
}

}  // namespace

extern "C" int b2_tfrecord_parse(b2_ctx* ctx, const uint8_t* shard, uint64_t nbytes, const uint64_t* rec_off,
                                 const uint64_t* rec_len, const b2_example_index* index, int n,
                                 uint64_t max_record_len, const b2_parse_sink* sink, int32_t* status,
                                 b2_stream stream) {
    B2_REQUIRE(ctx && shard && rec_off && rec_len && sink && status, "b2_tfrecord_parse: NULL argument");
    B2_REQUIRE(n >= 0 && n <= (1 << 24), "b2_tfrecord_parse: n out of range");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(shard) & 15) == 0, "b2_tfrecord_parse: shard must be 16-byte aligned");
    B2_REQUIRE(sink->mode == B2_SINK_NONE || index, "b2_tfrecord_parse: index required for a payload sink");
    if (int e = check_sink(sink, "b2_tfrecord_parse")) return e;
    if (n == 0) return 0;
    DeviceGuard g(ctx->device);
    ParseArgs pa = parse_args(ctx, shard, nbytes, rec_off, rec_len, index, *sink, status);
    return launch_uniform(ctx, pa, n, max_record_len, static_cast<cudaStream_t>(stream), "b2_tfrecord_parse");
}

extern "C" int b2_tfrecord_parse_table(b2_ctx* ctx, const uint8_t* shard, uint64_t nbytes, uint64_t max_records,
                                       uint8_t* table, const b2_parse_sink* sink, int32_t* status, b2_stream stream) {
    B2_REQUIRE(ctx && shard && table && sink && status, "b2_tfrecord_parse_table: NULL argument");
    B2_REQUIRE(max_records >= 1 && max_records <= (1u << 24), "b2_tfrecord_parse_table: max_records out of range");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(shard) & 15) == 0 && (reinterpret_cast<uintptr_t>(table) & 15) == 0,
               "b2_tfrecord_parse_table: shard and table must be 16-byte aligned");
    if (int e = check_sink(sink, "b2_tfrecord_parse_table")) return e;
    DeviceGuard g(ctx->device);
    const TableView v = table_view(table, nbytes, max_records);
    ParseArgs pa = parse_args(ctx, shard, nbytes, v.rec_off, v.rec_len, v.index, *sink, status);
    pa.tile2rec = v.tile2rec;
    pa.tile_start = v.tile_start;
    pa.hdr = v.hdr;
    pa.acc = v.acc;
    pa.n_bad = v.hdr + 4;
    pa.sched = reinterpret_cast<uint32_t*>(v.hdr + 5);
    pa.prof = dev_profile(ctx);
    pa.row_mask = dev_row_mask();
    return launch_fused(ctx, pa, v.cap_tiles, static_cast<cudaStream_t>(stream));
}

extern "C" int b2_crc32c(b2_ctx* ctx, const uint8_t* data, const uint64_t* offsets, const uint64_t* lens, int n,
                         uint64_t max_len, uint32_t* crc_out, b2_stream stream) {
    B2_REQUIRE(ctx && data && offsets && lens && crc_out, "b2_crc32c: NULL argument");
    B2_REQUIRE(n >= 0 && n <= (1 << 24), "b2_crc32c: n out of range");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(data) & 15) == 0, "b2_crc32c: data must be 16-byte aligned");
    if (n == 0) return 0;
    DeviceGuard g(ctx->device);
    b2_parse_sink sink{};   // B2_SINK_NONE: CRC only
    sink.verify_crc = 1;
    ParseArgs pa = parse_args(ctx, data, ~0ull, offsets, lens, nullptr, sink, nullptr);
    pa.crc_out = crc_out;
    return launch_uniform(ctx, pa, n, max_len, static_cast<cudaStream_t>(stream), "b2_crc32c");
}

#ifdef B2_DEV_KNOBS
/* development builds only (make DEV=1): with B2_PARSE_PROFILE set, b2_tfrecord_parse_table accumulates the cycles lane 0
 * of every warp spends in { tile wait, CRC, image sink, one-hot sink, end barrier, flush, job fetch, - } (out[0..7]: warp
 * 0, which also fetches the jobs; out[8..15]: the other warps); read and reset them here.  Not part of include/b2chips.h. */
extern "C" int b2_debug_parse_phases(b2_ctx* ctx, uint64_t out[16]) {
    B2_REQUIRE(ctx && out, "b2_debug_parse_phases: NULL argument");
    DeviceGuard g(ctx->device);
    B2_CUDA(cudaDeviceSynchronize());
    B2_CUDA(cudaMemcpy(out, ctx->prof_dev, 128, cudaMemcpyDeviceToHost));
    B2_CUDA(cudaMemset(ctx->prof_dev, 0, 128));
    return 0;
}
#endif
