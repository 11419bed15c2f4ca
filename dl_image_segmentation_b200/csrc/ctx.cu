// ctx.cu — context lifetime, error reporting, CRC-32C constant tables.
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace b2 {

static thread_local std::string g_err;

void set_error(const std::string& msg) { g_err = msg; }
int fail(const std::string& msg) {
    g_err = msg;
    return 1;
}
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return 2;
}

int ws_reserve(b2_ctx* ctx, size_t bytes, cudaStream_t s) {
    if (ctx->ws_used && ctx->ws_stream != s) {     // the previous user ran on another stream: wait for everything queued there
        B2_CUDA(cudaEventRecord(ctx->ws_event, ctx->ws_stream));
        B2_CUDA(cudaStreamWaitEvent(s, ctx->ws_event, 0));
    }
    ctx->ws_stream = s;
    ctx->ws_used = true;
    if (bytes <= ctx->ws_bytes) return 0;
    // growing is rare (first calls only); stream-ordered so in-flight users of the old block finish first
    if (ctx->ws) B2_CUDA(cudaFreeAsync(ctx->ws, s));
    ctx->ws = nullptr;
    ctx->ws_bytes = 0;
    size_t want = bytes + bytes / 2 + (1u << 16);
    B2_CUDA(cudaMallocAsync(&ctx->ws, want, s));
    ctx->ws_bytes = want;
    return 0;
}

// multiply by x^-1 in the reflected representation
static uint32_t div_x(uint32_t b) {
    uint32_t lsb = b >> 31;
    uint32_t t = b ^ (lsb ? kPoly : 0u);
    return (t << 1) | lsb;
}

static void build_tables(CrcTables* t) {
    uint32_t t0[256];
    for (uint32_t i = 0; i < 256; i++) {
        uint32_t c = i;
        for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ kPoly : (c >> 1);
        t0[i] = c;
    }
    auto adv1 = [&](uint32_t s) { return (s >> 8) ^ t0[s & 0xff]; };
    auto adv = [&](uint32_t s, int n) {
        for (int i = 0; i < n; i++) s = adv1(s);
        return s;
    };
    for (int k = 0; k < 4; k++)
        for (uint32_t v = 0; v < 256; v++) {
            t->t4[k][v] = adv(v << (8 * k), 4);
            t->s4096[k][v] = adv(v << (8 * k), 4 + 4096 - 16);
        }
    t->x2n[0] = 0x40000000u;  // x^1
    for (int k = 1; k < 64; k++) t->x2n[k] = multmodp(t->x2n[k - 1], t->x2n[k - 1]);
    const uint32_t xtile = t->x2n[16];    // x^(8*8192) = x^(2^16)
    t->tpow[0] = 0x80000000u;
    for (int j = 1; j < 2048; j++) t->tpow[j] = multmodp(t->tpow[j - 1], xtile);
    uint32_t xi8 = 0x80000000u;
    for (int k = 0; k < 8; k++) xi8 = div_x(xi8);      // x^-8
    uint32_t xi128 = xi8;
    for (int k = 0; k < 4; k++) xi128 = multmodp(xi128, xi128);  // x^-128
    uint32_t p = 0x80000000u;
    for (int r = 0; r < 16; r++) {
        t->xinvb[r] = p;
        p = multmodp(p, xi8);
    }
    p = 0x80000000u;
    for (int q = 0; q < 514; q++) {
        t->xinv16[q] = p;
        p = multmodp(p, xi128);
    }
}

}  // namespace b2

using namespace b2;

extern "C" {

int b2_version(void) { return B2_VERSION; }

const char* b2_last_error(void) { return g_err.c_str(); }

int b2_ctx_create(int device, b2_ctx** out) {
    B2_REQUIRE(out != nullptr, "b2_ctx_create: out is NULL");
    int count = 0;
    B2_CUDA(cudaGetDeviceCount(&count));
    B2_REQUIRE(device >= 0 && device < count, "b2_ctx_create: no such CUDA device");
    DeviceGuard g(device);
    B2_REQUIRE(g.ok, "b2_ctx_create: cannot select device");
    cudaDeviceProp prop;
    B2_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10 && !getenv("B2_ALLOW_ANY_ARCH"))
        return fail("b2_ctx_create: libb2chips is built for sm_100a (B200) only");
    b2_ctx* c = new b2_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->launches = 0;
    c->ws = nullptr;
    c->ws_bytes = 0;
    c->ws_mutex = new std::mutex();
    c->ws_stream = nullptr;
    c->ws_used = false;
    B2_CUDA(cudaEventCreateWithFlags(&c->ws_event, cudaEventDisableTiming));
    c->crc_host = new CrcTables();
    build_tables(c->crc_host);
    B2_CUDA(cudaMalloc(&c->crc_dev, sizeof(CrcTables)));
    B2_CUDA(cudaMemcpy(c->crc_dev, c->crc_host, sizeof(CrcTables), cudaMemcpyHostToDevice));
    B2_CUDA(cudaMalloc(&c->prof_dev, 128));
    B2_CUDA(cudaMemset(c->prof_dev, 0, 128));
    *out = c;
    return 0;
}

int b2_ctx_destroy(b2_ctx* ctx) {
    if (!ctx) return 0;
    DeviceGuard g(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->ws) cudaFree(ctx->ws);
    cudaEventDestroy(ctx->ws_event);
    delete ctx->ws_mutex;
    if (ctx->crc_dev) cudaFree(ctx->crc_dev);
    if (ctx->prof_dev) cudaFree(ctx->prof_dev);
    delete ctx->crc_host;
    delete ctx;
    return 0;
}

uint64_t b2_ctx_launch_count(const b2_ctx* ctx) { return ctx ? ctx->launches : 0; }
int b2_ctx_sm_count(const b2_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

}  // extern "C"
