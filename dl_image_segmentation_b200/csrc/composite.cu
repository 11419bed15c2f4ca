// composite.cu — K3: per-pixel compositors over a (T,H,W,B) time stack.
//
//   K3a  masked median            replaces np.ma.median(np.ma.masked_where(...), axis=0)
//                                 (_descartes_img_chips.py:562-567)
//   K3b  nearest-date mosaic      replaces filter + stable descending sort + SceneCollection.mosaic
//                                 (_descartes_img_chips.py:461-469, 603-626)
//
// Both are pure streaming kernels bounded by HBM bandwidth: every stack element is read exactly once
// (K3a) or at most once (K3b), straight from global memory with fully coalesced vector loads — there is
// no reuse, so no shared-memory staging.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "median_net.inc"

namespace b2 {

// ------------------------------------------------------------------------------------------------ K3a
//
// A thread owns ONE packed u16x2 register per scene = two consecutive bands of one pixel, and keeps the whole
// time series in registers (P slots, P = T rounded up to a power of two).  Invalid entries (cloud,
// nodata, or padding slots t >= T) are replaced by sentinels, alternating 0xFFFF, 0x0000, 0xFFFF ...
// per (pixel, band).  With m invalid entries that puts floor(m/2) zeros below and ceil(m/2) 0xFFFFs
// above the n = P - m valid values, so the valid values occupy ranks [floor(m/2), floor(m/2)+n) and their
// middle element(s) always sit at ranks P/2-1 (n odd) or P/2-1 and P/2 (n even).  Ties between a
// sentinel and a genuine 0 / 0xFFFF are harmless because equal keys are interchangeable.  A pruned
// selection network (median_net.inc) then extracts just those two ranks: no sort, no dynamic indexing.
//
// GPP = threads per pixel (B/2).  When it is a power of two the GPP threads of a pixel sit in one warp and
// SHARE the validity column: each loads P/GPP of the T bytes and the bit masks are OR-ed with warp shuffles,
// which removes (GPP-1)/GPP of the byte loads and their registers.  GPP = 0: every thread loads all T bytes.
// All loads of a thread are issued back to back before any is consumed (T + T/GPP independent requests).
// kFullT: T == P is known at compile time (the common case, e.g. T = 16), so no load or slot is predicated.
// Addresses advance by one scene plane per step (two adds) instead of being recomputed from t.
template <int P, int GPP, bool kNodata, bool kFullT>
__global__ void __launch_bounds__(256, (P <= 16 ? (kNodata ? 4 : 6) : 2))
median_kernel(const uint16_t* __restrict__ stack, const uint8_t* __restrict__ valid,
              const uint8_t* __restrict__ nodata, int T_rt, uint64_t hw, int B, uint64_t n_groups,
              double* __restrict__ out, uint8_t* __restrict__ out_mask) {
    const int T = kFullT ? P : T_rt;
    const uint64_t g_raw = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = g_raw < n_groups;
    const uint64_t g = live ? g_raw : n_groups - 1;   // keep every lane alive for the shuffles
    const uint64_t e0 = g * 2;                        // first element (pixel*B + band) of this thread
    const uint64_t pix = GPP ? g / GPP : e0 / (uint64_t)B;
    const uint64_t plane = hw * (uint64_t)B;          // elements per scene

    uint32_t v[P];
    {
        const uint8_t* p = reinterpret_cast<const uint8_t*>(stack + e0);
        const uint64_t step = plane * 2;
#pragma unroll
        for (int t = 0; t < P; t++) {
            v[t] = (kFullT || t < T) ? __ldg(reinterpret_cast<const uint32_t*>(p)) : 0u;
            p += step;
        }
    }
    uint32_t vmask = 0;                               // bit t set = scene t usable at this pixel
    if (GPP) {
        constexpr int kPer = GPP ? (P + GPP - 1) / GPP : P;
        const int sub = (int)(g % (GPP ? GPP : 1));
        uint32_t vb[kPer];
        const uint8_t* p = valid + (uint64_t)sub * hw + pix;
        const uint64_t step = (uint64_t)(GPP ? GPP : 1) * hw;
#pragma unroll
        for (int j = 0; j < kPer; j++) {
            const int t = sub + j * GPP;
            vb[j] = ((kFullT && (j + 1) * GPP <= P) || t < T) ? __ldg(p) : 0u;
            p += step;
        }
#pragma unroll
        for (int j = 0; j < kPer; j++) vmask |= (vb[j] ? 1u : 0u) << (j * GPP);
        vmask <<= sub;
#pragma unroll
        for (int o = 1; o < GPP; o <<= 1) vmask |= __shfl_xor_sync(0xffffffffu, vmask, o);
    } else {
        uint32_t vb[P];
        const uint8_t* p = valid + pix;
#pragma unroll
        for (int t = 0; t < P; t++) {
            vb[t] = (kFullT || t < T) ? __ldg(p) : 0u;
            p += hw;
        }
#pragma unroll
        for (int t = 0; t < P; t++) vmask |= (vb[t] ? 1u : 0u) << t;
    }
    uint32_t cnt;                                     // valid count per half
    if (kNodata) {
        uint32_t ndm[P];                              // per half 0xFFFF where the (t,band) sample is nodata
        const uint8_t* p = nodata + e0;
#pragma unroll
        for (int t = 0; t < P; t++) {
            const uint32_t two = (kFullT || t < T) ? __ldg(reinterpret_cast<const uint16_t*>(p)) : 0u;
            ndm[t] = ((two & 0xFFu) ? 0x0000FFFFu : 0u) | ((two & 0xFF00u) ? 0xFFFF0000u : 0u);
            p += plane;
        }
        uint32_t tg = 0xFFFFFFFFu;                    // next sentinel per half (0xFFFF first)
        cnt = 0;
#pragma unroll
        for (int t = 0; t < P; t++) {
            uint32_t im = ((vmask >> t) & 1u) ? 0u : 0xFFFFFFFFu;     // per half: 0xFFFF where the entry is invalid
            im |= ndm[t];
            v[t] = (v[t] & ~im) | (tg & im);
            tg ^= im;
            cnt += (~im) & 0x00010001u;
        }
    } else {
        // both halves share the validity: invalid entry number k gets the sentinel 0xFFFF (k even) or 0 (k odd);
        // slots t >= T are invalid too (their bits are 0 in vmask).  One bit test + two predicated moves per slot.
        uint32_t tg = 0xFFFFFFFFu;
#pragma unroll
        for (int t = 0; t < P; t++) {
            if (!((vmask >> t) & 1u)) {
                v[t] = tg;
                tg = ~tg;
            }
        }
        const uint32_t n = (uint32_t)__popc(vmask & (P < 32 ? ((1u << P) - 1u) : 0xFFFFFFFFu));
        cnt = n | (n << 16);
    }
    MedNet<P>::run(v);
    const uint32_t lo = v[P / 2 - 1], hi = v[P / 2];
    double res[2];
    uint32_t msk = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const uint32_t n = (cnt >> (16 * h)) & 0xFFFFu;
        const uint32_t a = (lo >> (16 * h)) & 0xFFFFu, b = (hi >> (16 * h)) & 0xFFFFu;
        // n odd -> the single middle (rank P/2-1); n even -> mean of the two middles
        const uint32_t sum2 = (n & 1u) ? 2u * a : a + b;
        // sum2 / 2 exactly, without an int->double conversion: 2^51 + sum2/2 is representable (ulp 0.5)
        res[h] = n ? __hiloint2double(0x43200000, (int)sum2) - 2251799813685248.0 : 0.0;
        msk |= (n ? 0u : 1u) << (8 * h);
    }
    if (live) {
        st_cs(reinterpret_cast<double2*>(out + e0), make_double2(res[0], res[1]));
        *reinterpret_cast<uint16_t*>(out_mask + e0) = (uint16_t)msk;
    }
}

// Generic fallback: any T, any B, one thread per (pixel, band); rank-counting selection straight from
// global memory (two passes over the series, no local arrays).  Used when T > 32 or B is odd.
__global__ void __launch_bounds__(256)
median_generic_kernel(const uint16_t* __restrict__ stack, const uint8_t* __restrict__ valid,
                      const uint8_t* __restrict__ nodata, int T, uint64_t hw, int B, uint64_t n_elems,
                      double* __restrict__ out, uint8_t* __restrict__ out_mask) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_elems) return;
    const uint64_t pix = e / (uint64_t)B;
    const uint64_t plane = hw * (uint64_t)B;
    int n = 0;
    for (int t = 0; t < T; t++) {
        bool ok = valid[(uint64_t)t * hw + pix] != 0;
        if (nodata) ok = ok && nodata[(uint64_t)t * plane + e] == 0;
        n += ok;
    }
    if (n == 0) {
        out[e] = 0.0;
        out_mask[e] = 1;
        return;
    }
    const int r_lo = (n - 1) / 2, r_hi = n / 2;
    uint32_t a = 0, b = 0;
    for (int t = 0; t < T; t++) {
        bool ok = valid[(uint64_t)t * hw + pix] != 0;
        if (nodata) ok = ok && nodata[(uint64_t)t * plane + e] == 0;
        if (!ok) continue;
        const uint32_t x = stack[(uint64_t)t * plane + e];
        int less = 0, leq = 0;  // rank interval of x among the valid values, ties broken by index
        for (int u = 0; u < T; u++) {
            bool ok2 = valid[(uint64_t)u * hw + pix] != 0;
            if (nodata) ok2 = ok2 && nodata[(uint64_t)u * plane + e] == 0;
            if (!ok2) continue;
            const uint32_t y = stack[(uint64_t)u * plane + e];
            less += (y < x) || (y == x && u < t);
            leq += 1;
        }
        (void)leq;
        if (less == r_lo) a = x;
        if (less == r_hi) b = x;
    }
    out[e] = 0.5 * (double)(a + b);
    out_mask[e] = 0;
}

template <int P, int GPP>
static void launch_median(const uint16_t* stack, const uint8_t* valid, const uint8_t* nodata, int T, uint64_t hw,
                          int B, double* out, uint8_t* mask, cudaStream_t s) {
    const uint64_t n_groups = hw * (uint64_t)B / 2;
    const unsigned grid = (unsigned)((n_groups + 255) / 256);
    if (nodata) {
        if (T == P) median_kernel<P, GPP, true, true><<<grid, 256, 0, s>>>(stack, valid, nodata, T, hw, B, n_groups, out, mask);
        else median_kernel<P, GPP, true, false><<<grid, 256, 0, s>>>(stack, valid, nodata, T, hw, B, n_groups, out, mask);
    } else {
        if (T == P) median_kernel<P, GPP, false, true><<<grid, 256, 0, s>>>(stack, valid, nodata, T, hw, B, n_groups, out, mask);
        else median_kernel<P, GPP, false, false><<<grid, 256, 0, s>>>(stack, valid, nodata, T, hw, B, n_groups, out, mask);
    }
}

template <int P>
static void dispatch_gpp(int gpp, const uint16_t* stack, const uint8_t* valid, const uint8_t* nodata, int T,
                         uint64_t hw, int B, double* out, uint8_t* mask, cudaStream_t s) {
    switch (gpp) {
        case 1: launch_median<P, 1>(stack, valid, nodata, T, hw, B, out, mask, s); break;
        case 2: launch_median<P, 2>(stack, valid, nodata, T, hw, B, out, mask, s); break;
        case 4: launch_median<P, 4>(stack, valid, nodata, T, hw, B, out, mask, s); break;
        case 8: launch_median<P, 8>(stack, valid, nodata, T, hw, B, out, mask, s); break;
        default: launch_median<P, 0>(stack, valid, nodata, T, hw, B, out, mask, s); break;
    }
}

static bool dispatch_median(int P, const uint16_t* stack, const uint8_t* valid, const uint8_t* nodata, int T,
                            uint64_t hw, int B, double* out, uint8_t* mask, cudaStream_t s) {
    const int gpp = B / 2;
    switch (P) {
        case 2: dispatch_gpp<2>(gpp, stack, valid, nodata, T, hw, B, out, mask, s); return true;
        case 4: dispatch_gpp<4>(gpp, stack, valid, nodata, T, hw, B, out, mask, s); return true;
        case 8: dispatch_gpp<8>(gpp, stack, valid, nodata, T, hw, B, out, mask, s); return true;
        case 16: dispatch_gpp<16>(gpp, stack, valid, nodata, T, hw, B, out, mask, s); return true;
        case 32: dispatch_gpp<32>(gpp, stack, valid, nodata, T, hw, B, out, mask, s); return true;
    }
    return false;
}

// ------------------------------------------------------------------------------------------------ K3b
//
// One CTA column per chip (blockIdx.y).  Prologue: the first T threads evaluate the search filter and
// rank the eligible scenes by (|day - ref| ascending, index descending) — the reverse of the painting
// order, so order[0] is the scene painted last, i.e. the one that wins wherever it is valid.
// Main loop: one thread per pixel walks `order`, probing one validity byte per scene (coalesced across
// the warp) and stops at the first valid scene; only that scene's pixel is read.  Filtered-out scenes
// are never touched, so the kernel moves far fewer bytes than the dense T-deep definition.
// kStats = element size (1 or 2 bytes) when the exact integer band statistics {n, sum x, lo, hi} (sum x^2 = lo + 2^16 hi) of the
// valid output pixels are accumulated in the same pass (B = PB / kStats <= 4 bands); 0 = no statistics.  Fusing them
// saves the separate statistics pass its re-read of the whole output.
//
// The prologue, shared by both mosaic kernels.  max_day == INT32_MAX means no upper bound, as min_day == INT32_MIN
// already means no lower one.  The distance is exact: |day - ref| < 2^32 fits a uint32_t, and eligibility is kept apart
// from it, so distances of 2^31 and more still rank by value.  Shared memory (mosaic_smem_bytes): dist[T] uint32,
// order[T] int32, elig[T] uint8.  Returns the number of eligible scenes; order[0, n) holds them, best first.
__host__ __device__ constexpr size_t mosaic_smem_bytes(int T) { return (size_t)T * (2 * sizeof(uint32_t) + 1); }

__device__ __forceinline__ int rank_scenes(uint32_t* sm, const int32_t* __restrict__ scene_day, const float* __restrict__ scene_cf,
                                           int32_t ref_day, int32_t min_day, int32_t max_day, float max_cf, int T) {
    uint32_t* dist = sm;
    int32_t* order = reinterpret_cast<int32_t*>(sm + T);
    uint8_t* elig = reinterpret_cast<uint8_t*>(sm + 2 * T);
    __shared__ int32_t n_el;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const int32_t d = scene_day[t];
        const float cf = scene_cf[t];
        bool ok = d >= min_day && (max_day == INT32_MAX || d < max_day);
        if (!isnan(max_cf)) ok = ok && (cf < max_cf);
        dist[t] = d >= ref_day ? (uint32_t)d - (uint32_t)ref_day : (uint32_t)ref_day - (uint32_t)d;
        elig[t] = ok;
    }
    if (threadIdx.x == 0) n_el = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        if (elig[t]) {
            const uint32_t k = dist[t];
            int r = 0;
            for (int u = 0; u < T; u++) {
                const uint32_t ku = dist[u];
                r += elig[u] && (ku < k || (ku == k && u > t));
            }
            order[r] = t;
            atomicAdd(&n_el, 1);
        }
    }
    __syncthreads();
    return n_el;
}

template <int PB, int kStats = 0>  // PB = bytes per pixel (all bands), 0 = runtime
__global__ void __launch_bounds__(256)
mosaic_kernel(const void* const* __restrict__ stacks, const uint8_t* const* __restrict__ valids,
              const int32_t* __restrict__ scene_day, const float* __restrict__ scene_cf, int32_t ref_day,
              int32_t min_day, int32_t max_day, float max_cf, int T, uint32_t hw, int pb_runtime,
              uint8_t* __restrict__ out, uint8_t* __restrict__ out_mask, int16_t* __restrict__ src_index,
              int32_t* __restrict__ n_eligible, unsigned long long* __restrict__ stats) {
    extern __shared__ uint32_t sm[];  // rank_scenes: dist[T], order[T], elig[T]
    const int32_t* order = reinterpret_cast<const int32_t*>(sm + T);
    const int chip = blockIdx.y;
    const int pb = PB ? PB : pb_runtime;
    const int ne = rank_scenes(sm, scene_day + (size_t)chip * T, scene_cf + (size_t)chip * T, ref_day, min_day, max_day, max_cf, T);
    if (n_eligible && blockIdx.x == 0 && threadIdx.x == 0) n_eligible[chip] = ne;
    const uint8_t* vchip = valids[chip];
    const uint8_t* schip = static_cast<const uint8_t*>(stacks[chip]);
    constexpr int kSB = kStats ? PB / (kStats ? kStats : 1) : 1;   // bands with fused statistics
    unsigned long long st_n = 0, st_s[kSB], st_q[kSB];
#pragma unroll
    for (int b = 0; b < kSB; b++) st_s[b] = st_q[b] = 0;
    // A pixel is a chain of dependent loads (validity of the best scene, of the next one ..., then the pixel itself), so a
    // thread keeps kMU pixels in flight: their validity probes of one scene are issued together, then their pixel loads.
    constexpr int kMU = 4;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t p0 = blockIdx.x * blockDim.x + threadIdx.x; p0 < hw; p0 += kMU * stride) {
        int sel[kMU];
        bool live[kMU];
#pragma unroll
        for (int u = 0; u < kMU; u++) {
            sel[u] = -1;
            live[u] = p0 + u * stride < hw;
        }
        for (int k = 0; k < ne; k++) {
            const int t = order[k];
            uint8_t v[kMU];
            bool open = false;
#pragma unroll
            for (int u = 0; u < kMU; u++) {
                v[u] = 0;
                if (live[u] && sel[u] < 0) {
                    v[u] = __ldg(vchip + (size_t)t * hw + (p0 + u * stride));
                    open = true;
                }
            }
            if (!open) break;
#pragma unroll
            for (int u = 0; u < kMU; u++)
                if (v[u]) sel[u] = t;
        }
        uint32_t w[kMU][4];                                        // the pixels' bytes (fast paths), for the statistics
#pragma unroll
        for (int u = 0; u < kMU; u++) {
            w[u][0] = w[u][1] = w[u][2] = w[u][3] = 0;
            if (!live[u] || sel[u] < 0) continue;
            const uint8_t* s = schip + ((size_t)sel[u] * hw + (p0 + u * stride)) * pb;
            if (PB == 16) { const uint4 q = __ldg(reinterpret_cast<const uint4*>(s)); w[u][0] = q.x; w[u][1] = q.y; w[u][2] = q.z; w[u][3] = q.w; }
            else if (PB == 8) { const uint2 q = __ldg(reinterpret_cast<const uint2*>(s)); w[u][0] = q.x; w[u][1] = q.y; }
            else if (PB == 4) w[u][0] = __ldg(reinterpret_cast<const uint32_t*>(s));
            else if (PB == 2) w[u][0] = __ldg(reinterpret_cast<const uint16_t*>(s));
        }
#pragma unroll
        for (int u = 0; u < kMU; u++) {
            if (!live[u]) continue;
            const uint32_t p = p0 + u * stride;
            uint8_t* o = out + ((size_t)chip * hw + p) * pb;
            if (PB == 16) *reinterpret_cast<uint4*>(o) = make_uint4(w[u][0], w[u][1], w[u][2], w[u][3]);
            else if (PB == 8) *reinterpret_cast<uint2*>(o) = make_uint2(w[u][0], w[u][1]);
            else if (PB == 4) *reinterpret_cast<uint32_t*>(o) = w[u][0];
            else if (PB == 2) *reinterpret_cast<uint16_t*>(o) = (uint16_t)w[u][0];
            else {
                const uint8_t* s = schip + ((size_t)(sel[u] < 0 ? 0 : sel[u]) * hw + p) * pb;
                for (int i = 0; i < pb; i++) o[i] = sel[u] < 0 ? (uint8_t)0 : s[i];
            }
            out_mask[(size_t)chip * hw + p] = sel[u] < 0;
            if (src_index) src_index[(size_t)chip * hw + p] = (int16_t)sel[u];
            if (kStats && sel[u] >= 0) {
                st_n++;
#pragma unroll
                for (int b = 0; b < kSB; b++) {
                    const unsigned long long x = kStats == 2 ? ((w[u][b >> 1] >> (16 * (b & 1))) & 0xFFFFu) : ((w[u][b >> 2] >> (8 * (b & 3))) & 0xFFu);
                    st_s[b] += x;
                    st_q[b] += x * x;
                }
            }
        }
    }
    if (kStats) {   // warp shuffle -> shared memory -> one 64-bit atomic per (CTA, band, counter)
        __shared__ unsigned long long red[8][2 * kSB + 1];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
        for (int o = 16; o; o >>= 1) st_n += __shfl_xor_sync(0xffffffffu, st_n, o);
        if (lane == 0) red[wid][2 * kSB] = st_n;
#pragma unroll
        for (int b = 0; b < kSB; b++) {
            unsigned long long sv = st_s[b], qv = st_q[b];
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                sv += __shfl_xor_sync(0xffffffffu, sv, o);
                qv += __shfl_xor_sync(0xffffffffu, qv, o);
            }
            if (lane == 0) {
                red[wid][b] = sv;
                red[wid][kSB + b] = qv;
            }
        }
        __syncthreads();
        if (threadIdx.x < kSB) {
            const int b = threadIdx.x;
            unsigned long long n = 0, sv = 0, qv = 0;
            for (int k = 0; k < 8; k++) {
                n += red[k][2 * kSB];
                sv += red[k][b];
                qv += red[k][kSB + b];
            }
            if (n) {
                atomicAdd(stats + 4 * b + 0, n);
                atomicAdd(stats + 4 * b + 1, sv);
                atomicAdd(stats + 4 * b + 2, qv & 0xFFFFull);
                atomicAdd(stats + 4 * b + 3, qv >> 16);
            }
        }
    }
}

// The same selection for 8-byte pixels (4 bands of uint16: BASELINE configs[4]) with FOUR ADJACENT pixels per thread and
// two such groups in flight: one 32-bit load brings the validity of a group for one scene (a warp covers 128 contiguous
// bytes instead of 32), the four pixels leave as two 16-byte stores, their mask as one 32-bit store.  The per-thread
// statistics are 32-bit sums folded into 64 bits once per chip (a thread sees at most hw / 256 pixels of 16 bits).
constexpr int kStatSlots = 256;

template <int kStats>   // 0: no statistics; 2: exact integer band statistics of uint16 pixels
__global__ void __launch_bounds__(256, kStats ? 4 : 2)   // the statistics variant must stay within 64 registers: 4 CTAs / SM
mosaic_vec8_kernel(const void* const* __restrict__ stacks, const uint8_t* const* __restrict__ valids,
                   const int32_t* __restrict__ scene_day, const float* __restrict__ scene_cf, int32_t ref_day, int32_t min_day,
                   int32_t max_day, float max_cf, int T, uint32_t hw, uint8_t* __restrict__ out, uint8_t* __restrict__ out_mask,
                   int16_t* __restrict__ src_index, int32_t* __restrict__ n_eligible, unsigned long long* __restrict__ stats) {
    extern __shared__ uint32_t sm[];  // rank_scenes: dist[T], order[T], elig[T]
    const int32_t* order = reinterpret_cast<const int32_t*>(sm + T);
    const int chip = blockIdx.y;
    const int ne = rank_scenes(sm, scene_day + (size_t)chip * T, scene_cf + (size_t)chip * T, ref_day, min_day, max_day, max_cf, T);
    if (n_eligible && blockIdx.x == 0 && threadIdx.x == 0) n_eligible[chip] = ne;
    const uint8_t* vchip = valids[chip];
    const uint2* schip = static_cast<const uint2*>(stacks[chip]);
    const bool v4 = (reinterpret_cast<uintptr_t>(vchip) & 3u) == 0;    // validity planes readable as 32-bit words
    uint32_t st_n = 0, st_s[4] = {0, 0, 0, 0};
    unsigned long long st_q[4] = {0, 0, 0, 0};
    constexpr int kG = 2;                                              // groups of 4 pixels in flight per thread
    const uint32_t groups = hw >> 2, stride = gridDim.x * blockDim.x;
    // validity word of one group for scene t
    auto vload = [&](int t, uint32_t g) -> uint32_t {
        const uint8_t* a = vchip + (size_t)t * hw + 4u * g;
        return v4 ? __ldg(reinterpret_cast<const uint32_t*>(a))
                  : ((uint32_t)__ldg(a) | ((uint32_t)__ldg(a + 1) << 8) | ((uint32_t)__ldg(a + 2) << 16) | ((uint32_t)__ldg(a + 3) << 24));
    };
    // the probes of the best scene for the NEXT round of groups are requested before this round's statistics are worked
    // out, so that the arithmetic hides behind them instead of delaying them
    uint32_t vfirst[kG];
#pragma unroll
    for (int u = 0; u < kG; u++) {
        const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x + u * stride;
        vfirst[u] = (ne > 0 && g < groups) ? vload(order[0], g) : 0u;
    }
    for (uint32_t g0 = blockIdx.x * blockDim.x + threadIdx.x; g0 < groups; g0 += kG * stride) {
        int sel[kG][4];
        uint32_t open[kG];                                             // bit j: pixel j of the group still unresolved
#pragma unroll
        for (int u = 0; u < kG; u++) {
            open[u] = (g0 + u * stride < groups) ? 0xFu : 0u;
#pragma unroll
            for (int j = 0; j < 4; j++) sel[u][j] = -1;
        }
        for (int k = 0; k < ne; k++) {
            uint32_t any_open = 0;
#pragma unroll
            for (int u = 0; u < kG; u++) any_open |= open[u];
            if (!any_open) break;
            const int t = order[k];
            uint32_t v[kG];
#pragma unroll
            for (int u = 0; u < kG; u++) {
                v[u] = 0;
                if (open[u]) v[u] = k == 0 ? vfirst[u] : vload(t, g0 + u * stride);
            }
#pragma unroll
            for (int u = 0; u < kG; u++)
#pragma unroll
                for (int j = 0; j < 4; j++)
                    if (((open[u] >> j) & 1u) && ((v[u] >> (8 * j)) & 0xFFu)) {
                        sel[u][j] = t;
                        open[u] &= ~(1u << j);
                    }
        }
        uint2 w[kG][4];
#pragma unroll
        for (int u = 0; u < kG; u++)
#pragma unroll
            for (int j = 0; j < 4; j++) {
                w[u][j] = make_uint2(0u, 0u);
                if (g0 + u * stride < groups && sel[u][j] >= 0)
                    w[u][j] = __ldg(schip + (size_t)sel[u][j] * hw + 4u * (g0 + u * stride) + j);
            }
#pragma unroll
        for (int u = 0; u < kG; u++) {
            const uint32_t gn = g0 + (kG + u) * stride;
            vfirst[u] = (ne > 0 && gn < groups) ? vload(order[0], gn) : 0u;
        }
#pragma unroll
        for (int u = 0; u < kG; u++) {
            const uint32_t g = g0 + u * stride;
            if (g >= groups) continue;
            const size_t p = (size_t)chip * hw + 4u * g;
            uint4* o = reinterpret_cast<uint4*>(out + p * 8);
            o[0] = make_uint4(w[u][0].x, w[u][0].y, w[u][1].x, w[u][1].y);
            o[1] = make_uint4(w[u][2].x, w[u][2].y, w[u][3].x, w[u][3].y);
            uint32_t m = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) m |= (sel[u][j] < 0 ? 1u : 0u) << (8 * j);
            *reinterpret_cast<uint32_t*>(out_mask + p) = m;
            if (src_index) {
                *reinterpret_cast<uint2*>(src_index + p) =
                    make_uint2(((uint32_t)sel[u][0] & 0xFFFFu) | ((uint32_t)sel[u][1] << 16), ((uint32_t)sel[u][2] & 0xFFFFu) | ((uint32_t)sel[u][3] << 16));
            }
            if (kStats) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    if (sel[u][j] < 0) continue;
                    st_n++;
                    const uint32_t x0 = w[u][j].x & 0xFFFFu, x1 = w[u][j].x >> 16, x2 = w[u][j].y & 0xFFFFu, x3 = w[u][j].y >> 16;
                    st_s[0] += x0; st_s[1] += x1; st_s[2] += x2; st_s[3] += x3;
                    st_q[0] += x0 * x0; st_q[1] += x1 * x1; st_q[2] += x2 * x2; st_q[3] += x3 * x3;
                }
            }
        }
    }
    if (kStats) {   // warp shuffle -> shared memory -> one 64-bit atomic per (CTA, band, counter)
        __shared__ unsigned long long red[8][9];
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        unsigned long long nn = st_n;
#pragma unroll
        for (int o = 16; o; o >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
        if (lane == 0) red[wid][8] = nn;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            unsigned long long sv = st_s[b], qv = st_q[b];
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                sv += __shfl_xor_sync(0xffffffffu, sv, o);
                qv += __shfl_xor_sync(0xffffffffu, qv, o);
            }
            if (lane == 0) {
                red[wid][b] = sv;
                red[wid][4 + b] = qv;
            }
        }
        __syncthreads();
        if (threadIdx.x < 4) {
            const int b = threadIdx.x;
            unsigned long long n = 0, sv = 0, qv = 0;
            for (int k = 0; k < 8; k++) {
                n += red[k][8];
                sv += red[k][b];
                qv += red[k][4 + b];
            }
            if (n) {   // thousands of CTAs adding to the same 16 words serialise in L2: each chip adds to one of kStatSlots copies
                unsigned long long* slot = stats + (size_t)(chip & (kStatSlots - 1)) * 12 + 3 * b;
                atomicAdd(slot + 0, n);
                atomicAdd(slot + 1, sv);
                atomicAdd(slot + 2, qv);
            }
        }
    }
}

// fold the slot copies into the caller's accumulators {n, sum x, lo, hi} per band (sum x^2 = lo + 2^16 hi, b2chips.h)
__global__ void stats_fold_kernel(const unsigned long long* __restrict__ slots, unsigned long long* __restrict__ stats) {
    const int b = threadIdx.x >> 5, lane = threadIdx.x & 31;       // one warp per band
    unsigned long long n = 0, sv = 0, qv = 0;
    for (int k = lane; k < kStatSlots; k += 32) {
        n += slots[(size_t)k * 12 + 3 * b + 0];
        sv += slots[(size_t)k * 12 + 3 * b + 1];
        qv += slots[(size_t)k * 12 + 3 * b + 2];
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        sv += __shfl_xor_sync(0xffffffffu, sv, o);
        qv += __shfl_xor_sync(0xffffffffu, qv, o);
    }
    if (lane == 0 && n) {
        atomicAdd(stats + 4 * b + 0, n);
        atomicAdd(stats + 4 * b + 1, sv);
        atomicAdd(stats + 4 * b + 2, qv & 0xFFFFull);
        atomicAdd(stats + 4 * b + 3, qv >> 16);
    }
}

}  // namespace b2

using namespace b2;

extern "C" int b2_median_composite_u16(b2_ctx* ctx, const uint16_t* stack, const uint8_t* valid, const uint8_t* nodata,
                                       int T, int H, int W, int B, double* out, uint8_t* out_mask, b2_stream stream) {
    B2_REQUIRE(ctx && stack && valid && out && out_mask, "b2_median_composite_u16: NULL argument");
    B2_REQUIRE(T >= 1 && H >= 1 && W >= 1 && B >= 1, "b2_median_composite_u16: T,H,W,B must be positive");
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint64_t hw = (uint64_t)H * W;
    int P = 2;
    while (P < T) P <<= 1;
    const bool aligned = (reinterpret_cast<uintptr_t>(stack) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0) &&
                         (reinterpret_cast<uintptr_t>(out_mask) % 4 == 0) &&
                         (!nodata || reinterpret_cast<uintptr_t>(nodata) % 4 == 0);
    bool done = false;
    if (P <= 32 && aligned && B % 2 == 0) done = dispatch_median(P, stack, valid, nodata, T, hw, B, out, out_mask, s);
    if (!done) {
        const uint64_t n = hw * (uint64_t)B;
        median_generic_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(stack, valid, nodata, T, hw, B, n, out, out_mask);
    }
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int b2_nearest_date_mosaic(b2_ctx* ctx, const void* const* stacks, const uint8_t* const* valids,
                                      const int32_t* scene_day, const float* scene_cf, int32_t ref_day,
                                      int32_t min_day, int32_t max_day, float max_cf, int n_chips, int T, int H,
                                      int W, int B, int elem_bytes, void* out, uint8_t* out_mask,
                                      int16_t* src_index, int32_t* n_eligible, uint64_t* stats_acc, b2_stream stream) {
    B2_REQUIRE(ctx && stacks && valids && scene_day && scene_cf && out && out_mask, "b2_nearest_date_mosaic: NULL argument");
    B2_REQUIRE(n_chips >= 1 && n_chips <= 65535, "b2_nearest_date_mosaic: n_chips must be in [1,65535] per call");
    B2_REQUIRE(T >= 1 && T <= 4096 && H >= 1 && W >= 1 && B >= 1, "b2_nearest_date_mosaic: bad T/H/W/B");
    B2_REQUIRE(elem_bytes == 1 || elem_bytes == 2 || elem_bytes == 4 || elem_bytes == 8,
               "b2_nearest_date_mosaic: elem_bytes must be 1, 2, 4 or 8");
    B2_REQUIRE((uint64_t)H * W < (1ull << 31), "b2_nearest_date_mosaic: chip too large");
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const uint32_t hw = (uint32_t)H * W;
    const int pb = B * elem_bytes;
    // enough CTAs per chip to fill the machine when n_chips is small, one per 1024 pixels at most
    unsigned per_chip = (hw + 1023) / 1024;
    const unsigned want = (unsigned)((ctx->sm_count * 8 + n_chips - 1) / n_chips);
    if (per_chip > want) per_chip = want > 0 ? want : 1;
    dim3 grid(per_chip, n_chips);
    const size_t smem = mosaic_smem_bytes(T);     // at most 36 KiB (T <= 4096): no opt-in needed
    const bool al = reinterpret_cast<uintptr_t>(out) % 16 == 0;  // each stack aligned to its pixel load: the caller's contract
#define B2_MOSAIC(PBV)                                                                                              \
    mosaic_kernel<PBV><<<grid, 256, smem, s>>>(stacks, valids, scene_day, scene_cf, ref_day, min_day, max_day, max_cf, \
                                               T, hw, pb, static_cast<uint8_t*>(out), out_mask, src_index, n_eligible, nullptr)
#define B2_MOSAIC_STATS(PBV, EB)                                                                                    \
    mosaic_kernel<PBV, EB><<<grid, 256, smem, s>>>(stacks, valids, scene_day, scene_cf, ref_day, min_day, max_day,  \
                                                   max_cf, T, hw, pb, static_cast<uint8_t*>(out), out_mask, src_index, \
                                                   n_eligible, reinterpret_cast<unsigned long long*>(stats_acc))
    const bool vec8 = al && pb == 8 && (hw & 3u) == 0 && reinterpret_cast<uintptr_t>(out_mask) % 4 == 0 &&
                      (!src_index || reinterpret_cast<uintptr_t>(src_index) % 8 == 0) && (!stats_acc || elem_bytes == 2) &&
                      hw / 256 < 60000;                                // 32-bit per-thread sums of 16-bit values
    if (vec8) {
        if (stats_acc) {
            const size_t slot_bytes = (size_t)kStatSlots * 12 * sizeof(unsigned long long);
            WsLock ws_lock(ctx);
            if (int e = ws_reserve(ctx, slot_bytes, s)) return e;
            B2_CUDA(cudaMemsetAsync(ctx->ws, 0, slot_bytes, s));
            unsigned long long* slots = static_cast<unsigned long long*>(ctx->ws);
            mosaic_vec8_kernel<2><<<grid, 256, smem, s>>>(stacks, valids, scene_day, scene_cf, ref_day, min_day, max_day, max_cf, T, hw,
                                                          static_cast<uint8_t*>(out), out_mask, src_index, n_eligible, slots);
            stats_fold_kernel<<<1, 128, 0, s>>>(slots, reinterpret_cast<unsigned long long*>(stats_acc));
            ctx->launches++;
        } else
            mosaic_vec8_kernel<0><<<grid, 256, smem, s>>>(stacks, valids, scene_day, scene_cf, ref_day, min_day, max_day, max_cf, T, hw,
                                                          static_cast<uint8_t*>(out), out_mask, src_index, n_eligible, nullptr);
    } else
    if (stats_acc) {
        B2_REQUIRE(al && (elem_bytes == 1 || elem_bytes == 2) && B <= 4 && (pb == 2 || pb == 4 || pb == 8),
                   "b2_nearest_date_mosaic: fused statistics need uint8 / uint16 chips of at most 4 bands, 2-, 4- or "
                   "8-byte pixels and a 16-byte aligned output (use b2_band_stats otherwise)");
        if (pb == 8 && elem_bytes == 2) B2_MOSAIC_STATS(8, 2);
        else if (pb == 4 && elem_bytes == 2) B2_MOSAIC_STATS(4, 2);
        else if (pb == 2 && elem_bytes == 2) B2_MOSAIC_STATS(2, 2);
        else if (pb == 4 && elem_bytes == 1) B2_MOSAIC_STATS(4, 1);
        else if (pb == 2 && elem_bytes == 1) B2_MOSAIC_STATS(2, 1);
        else return fail("b2_nearest_date_mosaic: fused statistics: unsupported pixel layout");
    } else
    if (al && pb == 16) B2_MOSAIC(16);
    else if (al && pb == 8) B2_MOSAIC(8);
    else if (al && pb == 4) B2_MOSAIC(4);
    else if (al && pb == 2) B2_MOSAIC(2);
    else B2_MOSAIC(0);
#undef B2_MOSAIC
#undef B2_MOSAIC_STATS
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}
