// tfrecord_common.cuh — device helpers shared by the TFRecord kernels (tfrecord.cu: scan / index / build;
// parse.cu: the fused CRC + payload pass).
#pragma once
#include "common.cuh"

namespace b2 {

struct CrcSmem {
    uint32_t t4[4][256];
    uint32_t s[4][256];
};

__device__ __forceinline__ uint32_t adv4(const uint32_t (*t)[256], uint32_t x) {
    return t[0][x & 0xff] ^ t[1][(x >> 8) & 0xff] ^ t[2][(x >> 16) & 0xff] ^ t[3][x >> 24];
}

__device__ __forceinline__ void load_crc_tables(CrcSmem* sm, const CrcTables* tab) {
    const uint32_t* g0 = &tab->t4[0][0];
    const uint32_t* g1 = &tab->s4096[0][0];
    uint32_t* d0 = &sm->t4[0][0];
    uint32_t* d1 = &sm->s[0][0];
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
        d0[i] = __ldg(g0 + i);
        d1[i] = __ldg(g1 + i);
    }
}

// zero the bytes of a 16-byte vector at absolute address a that fall outside [lo, hi)
__device__ __forceinline__ uint4 mask_vec(uint4 v, uint64_t a, uint64_t lo, uint64_t hi) {
    if (a >= lo && a + 16 <= hi) return v;
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint64_t p = a + 4 * q + j;
            if (p >= lo && p < hi) m |= 0xFFu << (8 * j);
        }
        w[q] &= m;
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// a(x)*b(x) mod P, fully unrolled and branch-free (5 instructions per bit instead of the rolled loop's 11)
__device__ __forceinline__ uint32_t multmodp_fast(uint32_t a, uint32_t b) {
    uint32_t p = 0;
#pragma unroll
    for (int k = 31; k >= 0; k--) {
        if (a & (1u << k)) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ kPoly : (b >> 1);
    }
    return p;
}

// 4 bytes at an arbitrary byte offset of a 4-byte aligned shared-memory buffer: two word loads + one funnel shift
__device__ __forceinline__ uint32_t smem_u32_unaligned(const uint32_t* buf32, uint32_t off) {
    const uint32_t w0 = buf32[off >> 2], w1 = buf32[(off >> 2) + 1];
    return __funnelshift_r(w0, w1, (off & 3) * 8);
}

// x^(8*n) mod P via the x^(2^k) table
__device__ inline uint32_t xpow8(const CrcTables* tab, uint64_t n) {
    uint32_t p = 0x80000000u;
    int k = 3;
    while (n) {
        if (n & 1) p = multmodp(__ldg(&tab->x2n[k & 63]), p);
        n >>= 1;
        k++;
    }
    return p;
}

// TFRecord's masked CRC, as stored in a frame's header and footer
__device__ __forceinline__ uint32_t mask_crc(uint32_t c) { return ((c >> 15) | (c << 17)) + 0xa282ead8u; }

// ---------------------------------------------------------------- record CRC-32C (reader: parse.cu, writer: build_kernel)
// A record's data CRC is computed over 8 KiB tiles on a 16-byte aligned grid, a run of consecutive tiles per CTA, without
// a CRC instruction.  The pure CRC (zero init) is linear over GF(2), so:
//   * bytes outside the record count as zero and the 0xFFFFFFFF init is XORed into its first four data bytes;
//   * thread i owns vectors i and i + 256 (16 bytes each) of every tile.  From the end of one of its vectors to the start
//     of its next one is always 4080 bytes, inside a tile and from one tile to the next, so one slice-by-4 step that
//     consumes 4 bytes and skips 4080 chains them all (crc_running_step) and the per-thread alignment (one GF(2)[x]
//     multiplication) is paid once per run of tiles, not once per tile;
//   * when a run ends, thread i's state sits 16 i bytes past the end of the run's last tile: multiplying by x^(-128 i)
//     aligns it and the lanes of a warp XOR together (crc_lane_partial); each kernel folds its warps in its own way;
//   * the run's partial moves to the end of the record's last tile and merges, with the run's tile count, into one
//     64-bit accumulator word per record, { CRC partial (low 32 bits) | tiles done (high 32) }, zero before the first
//     run (record_acc_merge);
//   * whoever completes the tile count un-advances the zero padding between the record end and the end of its last
//     tile and complements (record_crc).
// The grid is anchored at the aligned-down start of what a kernel stages: the record data for the reader (d0 & ~15), the
// frame for the writer ((d0 - 12) & ~15).  So the callers, not record_crc, know where the grid ends: they pass the padding.
// A record shorter than 4 bytes has no room for the init XOR: it carries no partial (crc_tiled) and record_crc takes
// its CRC bytewise.

// Whether a record of len data bytes carries a tiled CRC partial (else it is CRC'd bytewise when it completes)
__device__ __forceinline__ bool crc_tiled(uint64_t len) { return len >= 4; }

// One tile of a thread's running CRC state.  On return the state sits at (tile end + 16 i).
// ts = absolute start of the tile; [d0, d1) = the record's data; first = the tile holding d0; interior = no byte of the
// tile lies outside [d0, d1).
__device__ __forceinline__ uint32_t crc_running_step(uint32_t s, const uint4* buf4, const CrcSmem* cs, uint64_t ts, uint64_t d0,
                                                     uint64_t d1, bool first, bool interior) {
    const int i = threadIdx.x;
    uint4 v0 = buf4[i], v1 = buf4[i + 256];
    if (!interior) {
        v0 = mask_vec(v0, ts + 16ull * i, d0, d1);
        v1 = mask_vec(v1, ts + 4096 + 16ull * i, d0, d1);
        if (first && ts + 16ull * i + 16 > d0 && ts + 16ull * i < d0 + 4) {   // vectors touching the first four data bytes
            uint32_t w[4] = {v0.x, v0.y, v0.z, v0.w};
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint64_t p = ts + 16ull * i + 4 * q + k;
                    if (p >= d0 && p < d0 + 4) w[q] ^= 0xFFu << (8 * k);
                }
            v0 = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
    s = adv4(cs->t4, s ^ v0.x);
    s = adv4(cs->t4, s ^ v0.y);
    s = adv4(cs->t4, s ^ v0.z);
    s = adv4(cs->s, s ^ v0.w);
    s = adv4(cs->t4, s ^ v1.x);
    s = adv4(cs->t4, s ^ v1.y);
    s = adv4(cs->t4, s ^ v1.z);
    s = adv4(cs->s, s ^ v1.w);
    return s;
}

// x^(8*8192*j): advance a tile partial by j tiles
__device__ __forceinline__ uint32_t tile_power(const CrcTables* tab, uint32_t j) {
    return j < 2048 ? __ldg(&tab->tpow[j]) : xpow8(tab, (uint64_t)j * kTile);
}

// End of a run: align thread threadIdx.x's running state with the end of the run's last tile and XOR the warp's lanes
// together (every lane returns the warp's partial)
__device__ __forceinline__ uint32_t crc_lane_partial(const CrcTables* tab, uint32_t s) {
    uint32_t t = multmodp_fast(__ldg(&tab->xinv16[threadIdx.x]), s);
#pragma unroll
    for (int o = 16; o; o >>= 1) t ^= __shfl_xor_sync(0xffffffffu, t, o);
    return t;
}

// Merge a run into its record's accumulator word: the run's CTA-wide partial (at the end of the run's last tile) moves
// on by the tiles_after tiles that follow the run in the record, then `tiles` tiles are counted.  Returns the word after
// the merge: whoever sees the count complete finalises the record.  The XOR into the low word and the add to the high
// word are two atomics on ONE address, applied in program order, so whoever sees the count complete also sees every
// partial: no fence, no retry loop.
__device__ __forceinline__ unsigned long long record_acc_merge(const CrcTables* tab, unsigned long long* acc, uint32_t partial,
                                                               uint32_t tiles_after, uint32_t tiles) {
    if (partial) atomicXor(acc, (unsigned long long)multmodp_fast(tile_power(tab, tiles_after), partial));
    const unsigned long long add = (unsigned long long)tiles << 32;
    return atomicAdd(acc, add) + add;
}

// Bytewise CRC-32C of n bytes (init 0xFFFFFFFF, complemented)
__device__ __forceinline__ uint32_t crc_bytes(const CrcTables* tab, const uint8_t* p, uint64_t n) {
    uint32_t s = 0xFFFFFFFFu;
    for (uint64_t i = 0; i < n; i++) s = (s >> 8) ^ __ldg(&tab->t4[3][(s ^ p[i]) & 0xff]);
    return ~s;
}

// A completed record's unmasked CRC-32C.  acc: the low word of its accumulator (the partial at the end of its last tile);
// pad: the bytes from the record end to the end of its last tile; data, len: the record's bytes, read only when the
// record is too short to carry a partial.
__device__ __forceinline__ uint32_t record_crc(const CrcTables* tab, uint32_t acc, uint64_t pad, const uint8_t* data,
                                               uint64_t len) {
    if (!crc_tiled(len)) return crc_bytes(tab, data, len);
    acc = multmodp(__ldg(&tab->xinv16[pad >> 4]), acc);
    acc = multmodp(__ldg(&tab->xinvb[pad & 15]), acc);
    return ~acc;
}

// Masked CRC of a frame's 8 little-endian length bytes (the header CRC); t = byte table (t4[3], or a shared-memory copy)
__device__ __forceinline__ uint32_t crc_hdr8(uint64_t l, const uint32_t* t) {
    uint32_t s = 0xFFFFFFFFu;
#pragma unroll
    for (int i = 0; i < 8; i++) s = (s >> 8) ^ t[(s ^ (uint32_t)(l >> (8 * i))) & 0xff];
    return mask_crc(~s);
}

// little-endian integers at any byte address
__device__ __forceinline__ uint64_t rd_u64(const uint8_t* p) {
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) v |= (uint64_t)p[i] << (8 * i);
    return v;
}
__device__ __forceinline__ uint32_t rd_u32(const uint8_t* p) {
    uint32_t v = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) v |= (uint32_t)p[i] << (8 * i);
    return v;
}

// 16 bytes at shard + a (a is 16-aligned), zero beyond nbytes
__device__ __forceinline__ uint4 ld16_bounded(const uint8_t* shard, uint64_t a, uint64_t nbytes) {
    if (a + 16 <= nbytes) return ld_nc(reinterpret_cast<const uint4*>(shard + a));
    uint32_t w[4] = {0, 0, 0, 0};
    for (uint64_t p = a; p < nbytes; p++) w[(p - a) >> 2] |= (uint32_t)shard[p] << (8 * ((p - a) & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}
__host__ __device__ __forceinline__ uint32_t record_tiles(uint64_t d0, uint64_t len) {
    if (len == 0) return 1;                                  // an empty record still owns one (empty) tile
    return (uint32_t)((d0 + len - (d0 & ~15ull) + kTile - 1) / kTile);
}

// ---------------------------------------------------------------- shard table (b2_tfrecord_open / _parse_table)
// One caller-owned device buffer describing an opened shard; every section 16-byte aligned:
//   hdr int64[8]        [0] records  [1] scan status  [2] tiles  [3] longest record  [4] records with status != 0
//                       [5] chunk scheduler words of the fused pass
//   rec_off uint64[cap] | rec_len uint64[cap] | index b2_example_index[cap] | tile_start uint32[cap+1]
//   acc uint64[cap]                          (scratch of the fused pass: CRC partial | tiles done; zero between launches)
//   tile2rec uint32[cap_tiles]               (owner record of every 8 KiB tile)
struct TableView {
    int64_t* hdr;
    uint64_t* rec_off;
    uint64_t* rec_len;
    b2_example_index* index;
    uint32_t* tile_start;
    unsigned long long* acc;
    uint32_t* tile2rec;
    uint64_t cap, cap_tiles, bytes;
};
__host__ __device__ inline TableView table_view(uint8_t* t, uint64_t nbytes, uint64_t cap) {
    TableView v;
    auto up = [](uint64_t x) { return (x + 15) & ~15ull; };
    uint64_t o = 0;
    v.cap = cap;
    v.cap_tiles = nbytes / kTile + 2 * cap + 2;   // a record wastes at most two partial tiles
    v.hdr = reinterpret_cast<int64_t*>(t + o);             o += 64;
    v.rec_off = reinterpret_cast<uint64_t*>(t + o);        o += up(8 * cap);
    v.rec_len = reinterpret_cast<uint64_t*>(t + o);        o += up(8 * cap);
    v.index = reinterpret_cast<b2_example_index*>(t + o);  o += up(sizeof(b2_example_index) * cap);
    v.tile_start = reinterpret_cast<uint32_t*>(t + o);     o += up(4 * (cap + 1));
    v.acc = reinterpret_cast<unsigned long long*>(t + o);  o += up(8 * cap);
    v.tile2rec = reinterpret_cast<uint32_t*>(t + o);       o += up(4 * v.cap_tiles);
    v.bytes = o;
    return v;
}
__host__ __device__ inline uint64_t table_bytes(uint64_t nbytes, uint64_t cap) { return table_view(nullptr, nbytes, cap).bytes; }

}  // namespace b2
