// normalise.cu — K4: fused cast + per-band normalise + label one-hot, and exact integer band statistics.
//
// North-star row A17 (SURVEY.md section 8a).  Not present in the reference (nearest analogue: per-band-max display
// scaling, parse_tfrecords.ipynb cell 21); the definition is the oracle's (oracle/normalise.py):
//     x_hat = (float32(x) - mean[c]) / std[c]        IEEE float32 subtract and divide
//     onehot[..., k] = (label == k) ? 1.0f : 0.0f    out-of-range labels give an all-zero row (tf.one_hot)
// Both kernels are elementwise streams bounded by HBM bandwidth; they are write-dominated (4x and 4K x the
// input bytes), so every store is a coalesced 128-bit streaming store.
#include "common.cuh"

namespace b2 {

template <typename T>
__device__ __forceinline__ float to_f32(T v) { return (float)v; }

// four consecutive elements starting at element e0 (e0 % 4 == 0), as floats; one vector load when the base is aligned
template <typename T>
__device__ __forceinline__ void load4(const T* __restrict__ img, uint64_t e0, uint64_t n_elems, bool vec_ok, float (&x)[4]) {
    if (vec_ok && e0 + 4 <= n_elems) {
        if (sizeof(T) == 1) {
            const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(img + e0));
#pragma unroll
            for (int k = 0; k < 4; k++) x[k] = to_f32((T)((w >> (8 * k)) & 0xFFu));
        } else if (sizeof(T) == 2) {
            const uint2 w = __ldg(reinterpret_cast<const uint2*>(img + e0));
            x[0] = to_f32((T)(w.x & 0xFFFFu)); x[1] = to_f32((T)(w.x >> 16));
            x[2] = to_f32((T)(w.y & 0xFFFFu)); x[3] = to_f32((T)(w.y >> 16));
        } else {
            const uint4 w = __ldg(reinterpret_cast<const uint4*>(img + e0));
            x[0] = __uint_as_float(w.x); x[1] = __uint_as_float(w.y); x[2] = __uint_as_float(w.z); x[3] = __uint_as_float(w.w);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) x[k] = (e0 + k < n_elems) ? to_f32(img[e0 + k]) : 0.0f;
    }
}

// One thread per output float4 of the image: elements [4g, 4g+4) of the flattened (n_pixels*C) array.  The band of
// the first element advances by a constant per grid stride, so there is no division in the loop.
template <typename T>
__global__ void __launch_bounds__(256)
normalise_kernel(const T* __restrict__ img, const float* __restrict__ mean, const float* __restrict__ stdv,
                 uint64_t n_elems, int C, float* __restrict__ out) {
    __shared__ float s_mean[64], s_std[64];
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        s_mean[c] = mean[c];
        s_std[c] = stdv[c];
    }
    __syncthreads();
    const bool vec_ok = (reinterpret_cast<uintptr_t>(img) & (4 * sizeof(T) - 1)) == 0;
    const uint64_t groups = (n_elems + 3) >> 2;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c0 = (uint32_t)((4 * g) % (uint64_t)C);
    const uint32_t cstep = (uint32_t)((4 * stride) % (uint64_t)C);
    for (; g < groups; g += stride) {
        const uint64_t e0 = 4 * g;
        float x[4], f[4];
        load4<T>(img, e0, n_elems, vec_ok, x);
        uint32_t c = c0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            f[k] = __fdiv_rn(x[k] - s_mean[c], s_std[c]);
            c = (c + 1 == (uint32_t)C) ? 0 : c + 1;
        }
        if (e0 + 4 <= n_elems) {
            st_cs(reinterpret_cast<float4*>(out) + g, make_float4(f[0], f[1], f[2], f[3]));
        } else {
            for (uint64_t e = e0; e < n_elems; e++) out[e] = f[e - e0];
        }
        c0 += cstep;
        if (c0 >= (uint32_t)C) c0 -= (uint32_t)C;
    }
}

// One thread per output float4 of the one-hot tensor: floats [4g, 4g+4) of the flattened (n_pixels*K) array.  The
// (label, class) position of the first float advances by a constant per grid stride: no division in the loop.
template <typename L>
__global__ void __launch_bounds__(256)
onehot_kernel(const L* __restrict__ label, uint64_t n_pixels, int K, float* __restrict__ out) {
    const uint64_t n_fl = n_pixels * (uint64_t)K;
    const uint64_t groups = (n_fl + 3) >> 2;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t l0 = (4 * g) / (uint64_t)K;
    uint32_t c0 = (uint32_t)(4 * g - l0 * (uint64_t)K);
    const uint64_t lstep = (4 * stride) / (uint64_t)K;
    const uint32_t cstep = (uint32_t)(4 * stride - lstep * (uint64_t)K);
    for (; g < groups; g += stride) {
        const uint64_t f0 = 4 * g;
        uint64_t l = l0;
        uint32_t c = c0;
        float f[4];
        int cls = (l < n_pixels) ? label_class<L>(__ldg(label + l), K) : -1;   // -1 equals no class index
#pragma unroll
        for (int k = 0; k < 4; k++) {
            f[k] = (cls == (int)c) ? 1.0f : 0.0f;
            if (++c == (uint32_t)K) {
                c = 0;
                l++;
                if (k < 3) cls = (l < n_pixels) ? label_class<L>(__ldg(label + l), K) : -1;
            }
        }
        if (f0 + 4 <= n_fl) {
            st_cs(reinterpret_cast<float4*>(out) + g, make_float4(f[0], f[1], f[2], f[3]));
        } else {
            for (uint64_t e = f0; e < n_fl; e++) out[e] = f[e - f0];
        }
        l0 += lstep;
        c0 += cstep;
        if (c0 >= (uint32_t)K) {
            c0 -= (uint32_t)K;
            l0++;
        }
    }
}

// u8 images: the quotient (v - mean[c]) / std[c] takes 256 x C values, so a CTA tabulates them once (IEEE division,
// the same bits as the per-element kernel) and every element becomes one shared-memory lookup: the per-element kernel
// spends ~70 instructions per float4 on four divisions and is issue-bound at 60 % of HBM.
constexpr int kLutMaxC = 16;
__global__ void __launch_bounds__(256)
normalise_u8_lut_kernel(const uint8_t* __restrict__ img, const float* __restrict__ mean, const float* __restrict__ stdv,
                        uint64_t n_elems, int C, float* __restrict__ out) {
    extern __shared__ float lut[];                       // [C][256]
    for (int i = threadIdx.x; i < 256 * C; i += blockDim.x) {
        const int c = i >> 8, v = i & 255;
        lut[i] = __fdiv_rn((float)v - mean[c], stdv[c]);
    }
    __syncthreads();
    const bool vec_ok = (reinterpret_cast<uintptr_t>(img) & 3) == 0;
    const uint64_t groups = (n_elems + 3) >> 2;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c0 = (uint32_t)((4 * g) % (uint64_t)C);
    const uint32_t cstep = (uint32_t)((4 * stride) % (uint64_t)C);
    for (; g < groups; g += stride) {
        const uint64_t e0 = 4 * g;
        uint32_t w = 0;
        if (vec_ok && e0 + 4 <= n_elems) w = __ldg(reinterpret_cast<const uint32_t*>(img + e0));
        else
            for (int k = 0; k < 4; k++)
                if (e0 + k < n_elems) w |= (uint32_t)img[e0 + k] << (8 * k);
        float f[4];
        uint32_t c = c0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            f[k] = lut[(c << 8) + ((w >> (8 * k)) & 0xFFu)];
            c = (c + 1 == (uint32_t)C) ? 0 : c + 1;
        }
        if (e0 + 4 <= n_elems) {
            st_cs(reinterpret_cast<float4*>(out) + g, make_float4(f[0], f[1], f[2], f[3]));
        } else {
            for (uint64_t e = e0; e < n_elems; e++) out[e] = f[e - e0];
        }
        c0 += cstep;
        if (c0 >= (uint32_t)C) c0 -= (uint32_t)C;
    }
}

// One-hot through shared memory: a CTA owns 256 labels at a time, keeps their 256 x K floats (all zero) in shared
// memory, sets one 1.0f per valid label, streams the block out with coalesced 16-byte stores and clears its ones again.
// ~12 instructions per label instead of ~50 per float4: the per-float4 kernel is issue-bound at 60 % of HBM.
constexpr int kHotBlockMaxK = 24;                     // 2 x 256 x K floats <= 48 KiB of dynamic shared memory

template <typename L>
__global__ void __launch_bounds__(256)
onehot_block_kernel(const L* __restrict__ label, uint64_t n_pixels, int K, float* __restrict__ out) {
    extern __shared__ __align__(128) float blk_all[];    // two blocks of [256][K]: the bulk store of one overlaps the fill of the other
    const int tid = threadIdx.x;
    const uint32_t blk_fl = 256u * (uint32_t)K;
    for (uint32_t i = tid; i < 2 * blk_fl / 4; i += 256) reinterpret_cast<float4*>(blk_all)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    int old_k[2] = {-1, -1};                             // the one this thread left in each block
    __syncthreads();
    const uint64_t n_blocks = (n_pixels + 255) / 256;
    uint32_t it = 0;
    for (uint64_t b = blockIdx.x; b < n_blocks; b += gridDim.x, it++) {
        const int sl = (int)(it & 1u);
        float* blk = blk_all + (size_t)sl * blk_fl;
        const uint64_t base = b * 256;
        const uint32_t n = (uint32_t)min((uint64_t)256, n_pixels - base);
        int k = -1;
        if ((uint32_t)tid < n) k = label_class<L>(__ldg(label + base + tid), K);
        if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the store that last used this block has read it
        __syncthreads();
        const int ok = sl ? old_k[1] : old_k[0];
        if (ok >= 0) blk[tid * K + ok] = 0.0f;
        if (k >= 0) blk[tid * K + k] = 1.0f;
        if (sl) old_k[1] = k; else old_k[0] = k;
        float* dst = out + base * (uint64_t)K;           // base * K * 4 bytes: a multiple of 1024
        const uint32_t n_fl = n * (uint32_t)K;
        if (n == 256) {                                  // whole block: one TMA bulk store, issued by one thread
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
                             "r"((uint32_t)__cvta_generic_to_shared(blk)), "r"(n_fl * 4u) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        } else {                                         // the ragged last block: plain stores
            __syncthreads();
            for (uint32_t i = tid; i < n_fl / 4; i += 256) st_cs(reinterpret_cast<float4*>(dst) + i, reinterpret_cast<const float4*>(blk)[i]);
            for (uint32_t i = (n_fl & ~3u) + tid; i < n_fl; i += 256) dst[i] = blk[i];
        }
    }
    if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");       // shared memory must outlive the bulk stores
    __syncthreads();
}

// Band statistics.  Thread-private 64-bit accumulators per band, warp-shuffle + shared-memory reduction, then one
// 64-bit atomic per (CTA, band, counter).  x*x is split at bit 16 so that the global accumulators cannot overflow
// 2^64 for any realistic dataset (SURVEY.md section 8e).  kB = compile-time band count (0 = runtime, up to kMaxB):
// with kB known the pixel is fetched with ONE vector load and the accumulators stay in a few registers.
constexpr int kMaxB = 16;

template <typename T, int kB>
__global__ void __launch_bounds__(256)
stats_kernel(const T* __restrict__ img, const uint8_t* __restrict__ valid, uint64_t n_pixels, int B_rt,
             unsigned long long* __restrict__ acc) {
    constexpr int NB = kB ? kB : kMaxB;
    const int B = kB ? kB : B_rt;
    unsigned long long cnt = 0, sum[NB], sq[NB];
#pragma unroll
    for (int b = 0; b < NB; b++) sum[b] = sq[b] = 0;
    constexpr int PB = kB * (int)sizeof(T);                               // bytes per pixel when known
    const bool vec_ok = kB && (PB == 2 || PB == 4 || PB == 8 || PB == 16) && (reinterpret_cast<uintptr_t>(img) % (PB ? PB : 1)) == 0;
    // Fast path: every pixel counts and a pixel is 2..16 bytes: 16 bytes (1..8 pixels) per load, sums of x in 32 bits (folded
    // into the 64-bit totals every 4096 loads: 4096 * 8 * 65535 < 2^32), x*x through one 32x32->64 multiply-add each.
    if (vec_ok && !valid && (reinterpret_cast<uintptr_t>(img) & 15) == 0) {
        constexpr int PPL = PB ? 16 / PB : 1;                               // pixels per 16-byte load
        const uint64_t n_vec = n_pixels / PPL;
        uint32_t s32[NB];
#pragma unroll
        for (int b = 0; b < NB; b++) s32[b] = 0;
        uint32_t since = 0;
        for (uint64_t v = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += (uint64_t)gridDim.x * blockDim.x) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(img) + v);
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int i = 0; i < PPL; i++) {
#pragma unroll
                for (int b = 0; b < NB; b++) {
                    const int e = i * NB + b;                               // sample index inside the 16 bytes
                    const uint32_t x = sizeof(T) == 2 ? ((w[e >> 1] >> (16 * (e & 1))) & 0xFFFFu) : ((w[e >> 2] >> (8 * (e & 3))) & 0xFFu);
                    s32[b] += x;
                    sq[b] += (unsigned long long)x * x;
                }
            }
            cnt += PPL;
            if (++since == 4096) {
#pragma unroll
                for (int b = 0; b < NB; b++) { sum[b] += s32[b]; s32[b] = 0; }
                since = 0;
            }
        }
#pragma unroll
        for (int b = 0; b < NB; b++) sum[b] += s32[b];
        // the pixels that do not fill a vector
        for (uint64_t p = n_vec * PPL + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pixels; p += (uint64_t)gridDim.x * blockDim.x) {
            cnt++;
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const unsigned long long x = (unsigned long long)img[p * (uint64_t)NB + b];
                sum[b] += x;
                sq[b] += x * x;
            }
        }
    } else
    for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pixels; p += (uint64_t)gridDim.x * blockDim.x) {
        if (valid && !valid[p]) continue;
        cnt++;
        if (vec_ok) {
            uint32_t w[4] = {0, 0, 0, 0};
            const uint8_t* px = reinterpret_cast<const uint8_t*>(img) + p * (uint64_t)PB;
            if (PB == 16) { const uint4 v = __ldg(reinterpret_cast<const uint4*>(px)); w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; }
            else if (PB == 8) { const uint2 v = __ldg(reinterpret_cast<const uint2*>(px)); w[0] = v.x; w[1] = v.y; }
            else if (PB == 4) w[0] = __ldg(reinterpret_cast<const uint32_t*>(px));
            else w[0] = __ldg(reinterpret_cast<const uint16_t*>(px));
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const unsigned long long x = sizeof(T) == 2 ? ((w[b >> 1] >> (16 * (b & 1))) & 0xFFFFu) : ((w[b >> 2] >> (8 * (b & 3))) & 0xFFu);
                sum[b] += x;
                sq[b] += x * x;
            }
        } else {
            const T* px = img + p * (uint64_t)B;
#pragma unroll
            for (int b = 0; b < NB; b++) {
                if (b < B) {
                    const unsigned long long x = (unsigned long long)px[b];
                    sum[b] += x;
                    sq[b] += x * x;
                }
            }
        }
    }
    __shared__ unsigned long long red[8][2 * NB + 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) red[wid][2 * NB] = cnt;
#pragma unroll
    for (int b = 0; b < NB; b++) {
        if (b < B) {
            unsigned long long sv = sum[b], q = sq[b];
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                sv += __shfl_xor_sync(0xffffffffu, sv, o);
                q += __shfl_xor_sync(0xffffffffu, q, o);
            }
            if (lane == 0) {
                red[wid][b] = sv;
                red[wid][NB + b] = q;
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < B) {
        const int b = threadIdx.x;
        unsigned long long n = 0, sv = 0, q = 0;
        for (int w = 0; w < 8; w++) {
            n += red[w][2 * NB];
            sv += red[w][b];
            q += red[w][NB + b];
        }
        // per-CTA q < 2^64 is guaranteed (<= 2^32 per pixel, a CTA sees far fewer than 2^32 pixels)
        atomicAdd(acc + 4 * b + 0, n);
        atomicAdd(acc + 4 * b + 1, sv);
        atomicAdd(acc + 4 * b + 2, q & 0xFFFFull);
        atomicAdd(acc + 4 * b + 3, q >> 16);
    }
}

}  // namespace b2

using namespace b2;

static unsigned stream_grid(const b2_ctx* ctx, uint64_t items) {
    uint64_t blocks = (items + 255) / 256;
    const uint64_t cap = (uint64_t)ctx->sm_count * 32;  // several waves of resident CTAs, grid-stride beyond
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks ? blocks : 1);
}

extern "C" int b2_normalise_onehot(b2_ctx* ctx, const void* img, int img_dtype, const void* label, int label_dtype,
                                   const float* mean, const float* stdv, uint64_t n_pixels, int C, int K,
                                   float* img_out, float* onehot_out, b2_stream stream) {
    B2_REQUIRE(ctx, "b2_normalise_onehot: NULL ctx");
    B2_REQUIRE(!img_out || (img && mean && stdv && C >= 1 && C <= 64), "b2_normalise_onehot: image path needs img, mean, std, 1<=C<=64");
    B2_REQUIRE(!onehot_out || (label && K >= 1), "b2_normalise_onehot: one-hot path needs label and K>=1");
    B2_REQUIRE((reinterpret_cast<uintptr_t>(img_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(onehot_out) & 15) == 0,
               "b2_normalise_onehot: outputs must be 16-byte aligned");
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (img_out && n_pixels) {
        const uint64_t n = n_pixels * (uint64_t)C;
        const unsigned grid = stream_grid(ctx, (n + 3) / 4);
        switch (img_dtype) {
            case B2_U8:
                if (C <= kLutMaxC)
                    normalise_u8_lut_kernel<<<grid, 256, (size_t)C * 256 * sizeof(float), s>>>(static_cast<const uint8_t*>(img), mean, stdv, n, C, img_out);
                else
                    normalise_kernel<uint8_t><<<grid, 256, 0, s>>>(static_cast<const uint8_t*>(img), mean, stdv, n, C, img_out);
                break;
            case B2_U16: normalise_kernel<uint16_t><<<grid, 256, 0, s>>>(static_cast<const uint16_t*>(img), mean, stdv, n, C, img_out); break;
            case B2_I16: normalise_kernel<int16_t><<<grid, 256, 0, s>>>(static_cast<const int16_t*>(img), mean, stdv, n, C, img_out); break;
            case B2_F32: normalise_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(img), mean, stdv, n, C, img_out); break;
            default: return fail("b2_normalise_onehot: img_dtype must be u8, u16, i16 or f32");
        }
        ctx->launches++;
        B2_CUDA(cudaGetLastError());
    }
    if (onehot_out && n_pixels) {
        const unsigned grid = stream_grid(ctx, (n_pixels * (uint64_t)K + 3) / 4);
        const bool blocks = K <= kHotBlockMaxK;          // 256 x K floats of shared memory per CTA
        unsigned bgrid = (unsigned)min((uint64_t)ctx->sm_count * (K <= 12 ? 8u : 3u), (n_pixels + 255) / 256);
        if (bgrid < 1) bgrid = 1;
        const size_t bsm = (size_t)2 * 256 * K * sizeof(float);
        if (label_dtype == B2_U8) {
            if (blocks) onehot_block_kernel<uint8_t><<<bgrid, 256, bsm, s>>>(static_cast<const uint8_t*>(label), n_pixels, K, onehot_out);
            else onehot_kernel<uint8_t><<<grid, 256, 0, s>>>(static_cast<const uint8_t*>(label), n_pixels, K, onehot_out);
        } else if (label_dtype == B2_F32) {
            if (blocks) onehot_block_kernel<float><<<bgrid, 256, bsm, s>>>(static_cast<const float*>(label), n_pixels, K, onehot_out);
            else onehot_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(label), n_pixels, K, onehot_out);
        } else {
            return fail("b2_normalise_onehot: label_dtype must be u8 or f32");
        }
        ctx->launches++;
        B2_CUDA(cudaGetLastError());
    }
    return 0;
}

extern "C" int b2_band_stats(b2_ctx* ctx, const void* img, int dtype, const uint8_t* valid, uint64_t n_pixels, int B,
                             uint64_t* acc, b2_stream stream) {
    B2_REQUIRE(ctx && img && acc, "b2_band_stats: NULL argument");
    B2_REQUIRE(B >= 1 && B <= kMaxB, "b2_band_stats: 1 <= B <= 16");
    if (n_pixels == 0) return 0;
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const unsigned grid = stream_grid(ctx, n_pixels);
    unsigned long long* a = reinterpret_cast<unsigned long long*>(acc);
#define B2_STATS(TY, KB) stats_kernel<TY, KB><<<grid, 256, 0, s>>>(static_cast<const TY*>(img), valid, n_pixels, B, a)
    if (dtype == B2_U8) {
        if (B == 2) B2_STATS(uint8_t, 2); else if (B == 4) B2_STATS(uint8_t, 4); else if (B == 8) B2_STATS(uint8_t, 8);
        else B2_STATS(uint8_t, 0);
    } else if (dtype == B2_U16) {
        if (B == 1) B2_STATS(uint16_t, 1); else if (B == 2) B2_STATS(uint16_t, 2); else if (B == 4) B2_STATS(uint16_t, 4);
        else if (B == 8) B2_STATS(uint16_t, 8); else B2_STATS(uint16_t, 0);
    } else {
        return fail("b2_band_stats: dtype must be u8 or u16");
    }
#undef B2_STATS
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}
