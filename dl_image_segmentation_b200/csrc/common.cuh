// common.cuh — context, error plumbing and small device helpers shared by all kernels of libb2chips.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>
#include <string>

#include "../../include/b2chips.h"

namespace b2 {

// ---------------------------------------------------------------- CRC-32C constant tables (device, per ctx)
struct CrcTables {
    uint32_t t4[4][256];     // standard slice-by-4: t4[k][v] = state v<<(8k) advanced by 4 zero bytes
    uint32_t s4096[4][256];  // same, advanced by 4 + 4096 - 16 bytes (second vector of a thread in a 8 KiB tile)
    uint32_t fix[256];       // fix[i] = x^(-128 i): undo the 16*i byte over-advance of thread i
    uint32_t xinv16[514];    // xinv16[q] = x^(-128 q): un-advance by q 16-byte vectors (tile padding)
    uint32_t xinvb[16];      // xinvb[r]  = x^(-8 r)
    uint32_t x2n[64];        // x^(2^k) for x2n pow
    uint32_t xtile;          // x^(8*8192): advance by one tile
    uint32_t tpow[2048];     // tpow[j] = x^(8*8192*j): advance by j tiles (records up to 16 MiB; beyond -> xpow8)
};

}  // namespace b2

struct b2_ctx {
    int device;
    int sm_count;
    uint64_t launches;
    b2::CrcTables* crc_dev;  // device copy
    b2::CrcTables* crc_host;
    unsigned long long* prof_dev;  // 8 phase counters (b2_debug_parse_phases)
    void* ws;                // grow-on-demand workspace, shared by the entry points that need scratch (see WsLock)
    size_t ws_bytes;
    std::mutex* ws_mutex;    // one workspace user at a time on the host ...
    cudaStream_t ws_stream;  // ... and on the device: the stream of the last user,
    cudaEvent_t ws_event;    //     which the next user's stream waits for when it is a different one
    bool ws_used;
};

namespace b2 {

void set_error(const std::string& msg);
int fail(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what);
int ws_reserve(b2_ctx* ctx, size_t bytes, cudaStream_t s);

// Entry points that use the context workspace hold this for their whole body: calls on one context from several host
// threads take turns, and ws_reserve orders a call behind the previous user's work when that ran on another stream, so two
// streams never have kernels in flight on the same scratch (ADVICE r1: the rule used to be a comment).
struct WsLock {
    std::lock_guard<std::mutex> g;
    explicit WsLock(b2_ctx* ctx) : g(*ctx->ws_mutex) {}
};

#define B2_CUDA(expr)                                            \
    do {                                                         \
        cudaError_t _e = (expr);                                 \
        if (_e != cudaSuccess) return b2::cuda_fail(_e, #expr);  \
    } while (0)

#define B2_REQUIRE(cond, msg)                 \
    do {                                      \
        if (!(cond)) return b2::fail(msg);    \
    } while (0)

// RAII device guard so that entry points work whatever device the caller has current
struct DeviceGuard {
    int prev;
    bool ok;
    explicit DeviceGuard(int dev) : prev(-1), ok(true) {
        if (cudaGetDevice(&prev) != cudaSuccess) ok = false;
        if (ok && prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() {
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && cur != prev && prev >= 0) cudaSetDevice(prev);
    }
};

constexpr uint32_t kPoly = 0x82F63B78u;  // CRC-32C (Castagnoli), reflected
constexpr int kTile = 8192;              // bytes of record data per CTA tile
constexpr int kTileThreads = 256;

// a(x)*b(x) mod P in the reflected representation (bit 31 = x^0)
__host__ __device__ inline uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
#pragma unroll 1
    for (uint32_t m = 0x80000000u; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ kPoly : (b >> 1);
    }
    return p;
}

// streaming (evict-first) 128-bit store for write-once outputs
__device__ __forceinline__ void st_cs(float4* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_cs(uint4* p, uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_cs(double2* p, double2 v) {
    asm volatile("st.global.cs.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}
// read-once 128-bit load that does not pollute L1
__device__ __forceinline__ uint4 ld_nc(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// The class of a label, or -1 for an all-zero one-hot row: the value must equal an integer k < K.  NaN, +-inf,
// negative and non-integral labels have no class; -0.0 is class 0.  The standalone one-hot (normalise.cu) and the
// fused parse (parse.cu) both ask here, so the two cannot diverge.
template <typename L>
__device__ __forceinline__ int label_class(L lab, int K);
template <>
__device__ __forceinline__ int label_class<uint8_t>(uint8_t lab, int K) { return (int)lab < K ? (int)lab : -1; }
template <>
__device__ __forceinline__ int label_class<float>(float lab, int K) {
    if (!(lab >= 0.0f && lab < 2147483648.0f)) return -1;  // also rejects NaN; below 2^31 the int conversion is exact
    const int k = (int)lab;
    return (float)k == lab && k < K ? k : -1;             // k < K in integers: (float)K would round above 2^24
}

}  // namespace b2
