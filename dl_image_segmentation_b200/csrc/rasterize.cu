// rasterize.cu — label rasterisation: polygons -> (H, W) uint8 with GDAL's ALL_TOUCHED semantics.
//
// Replaces gdal.RasterizeLayer(mem_ds, [1], layer, options=['ALL_TOUCHED=TRUE'[, 'ATTRIBUTE=...']]) on a background-filled
// Byte raster, create_label_array_for_tile (_descartes_img_chips.py:633-689).  GDAL burns feature after feature, so a pixel
// shared by several polygons keeps the value of the LAST one (the reference's comment, :676-683); here every burn is an
// atomicMax of the feature's index into a per-pixel owner word and one last pass turns owners into values: the same
// result whatever the order the threads run in.  Two burn passes per feature, as in GDAL's alg/llrasterize.cpp:
//   fill  (GDALdllImageFilledPolygon): one thread per (feature, scanline): crossings of the pixel-centre line y + 0.5 with
//         every edge (half-open in y), rounded floor(x + 0.5), sorted, spans between pairs burnt (even-odd rule);
//   lines (GDALdllImageLineAllTouched): one thread per edge, stepping from pixel boundary to pixel boundary.
// All coordinate arithmetic is IEEE double with explicit round-to-nearest operations (no fused multiply-add), in the
// order oracle/rasterize.py states it, so the burnt set is bit-identical with the CPU restatement.
// Label layers in another CRS than the tile's are brought into it first, vertex by vertex (project_points_kernel).
#include <math_constants.h>

#include "common.cuh"

namespace b2 {
namespace {

__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

__device__ __forceinline__ void burn(int32_t* owner, int W, int y, int x, int f) { atomicMax(owner + (size_t)y * W + x, f); }

// which feature does job / segment `i` belong to: last f with off[f] <= i
__device__ __forceinline__ int find_owner(const uint32_t* __restrict__ off, int n, uint32_t i) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(128)
raster_fill_kernel(const double4* __restrict__ segs, const uint32_t* __restrict__ seg_off, const int32_t* __restrict__ feat_miny,
                   const uint32_t* __restrict__ job_off, int n_features, uint32_t n_jobs, int W, int H,
                   const uint64_t* __restrict__ job_ints_off, int32_t* __restrict__ ints_ws, int32_t* __restrict__ owner) {
    const uint32_t job = blockIdx.x * blockDim.x + threadIdx.x;
    if (job >= n_jobs) return;
    const int f = find_owner(job_off, n_features, job);
    const int y = feat_miny[f] + (int)(job - job_off[f]);
    const double dy = (double)y + 0.5;
    int32_t* ints = ints_ws + job_ints_off[job];
    const uint32_t cap = (uint32_t)(job_ints_off[job + 1] - job_ints_off[job]);
    uint32_t n = 0;
    for (uint32_t s = seg_off[f]; s < seg_off[f + 1]; s++) {
        const double4 e = segs[s];                                   // (x1, y1) -> (x2, y2), ind1 = the earlier vertex
        double dy1 = e.y, dy2 = e.w, dx1, dx2;
        if ((dy1 < dy && dy2 < dy) || (dy1 > dy && dy2 > dy)) continue;
        if (dy1 < dy2) { dx1 = e.x; dx2 = e.z; }
        else if (dy1 > dy2) { dy2 = e.y; dy1 = e.w; dx2 = e.x; dx1 = e.z; }
        else {                                                       // the edge lies on the centre line
            if (e.x > e.z) {
                const int hx1 = (int)floor(dadd(e.z, 0.5)), hx2 = (int)floor(dadd(e.x, 0.5));
                if (!(hx1 > W - 1 || hx2 <= 0))
                    for (int x = max(hx1, 0); x <= min(hx2 - 1, W - 1); x++) burn(owner, W, y, x, f);
            }
            continue;
        }
        if (dy < dy2 && dy >= dy1) {
            const double inter = dadd(ddiv(dmul(dsub(dy, dy1), dsub(dx2, dx1)), dsub(dy2, dy1)), dx1);
            if (n < cap) ints[n] = (int)floor(dadd(inter, 0.5));
            n++;
        }
    }
    if (n > cap) n = cap;                                            // cannot happen: cap >= the edges this row can cross
    for (uint32_t i = 1; i < n; i++) {                               // crossings per scanline are few: insertion sort
        const int32_t v = ints[i];
        uint32_t j = i;
        while (j > 0 && ints[j - 1] > v) { ints[j] = ints[j - 1]; j--; }
        ints[j] = v;
    }
    for (uint32_t i = 0; i + 1 < n; i += 2) {
        const int a = ints[i], b = ints[i + 1];
        if (a <= W - 1 && b > 0)
            for (int x = max(a, 0); x <= min(b - 1, W - 1); x++) burn(owner, W, y, x, f);
    }
}

__global__ void __launch_bounds__(128)
raster_lines_kernel(const double4* __restrict__ segs, const uint32_t* __restrict__ seg_feat, uint32_t n_segs, int W, int H,
                    int32_t* __restrict__ owner) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_segs) return;
    const double4 e = segs[s];
    const int f = (int)seg_feat[s];
    double x = e.x, y = e.y, xe = e.z, ye = e.w;
    const double dW = (double)W, dH = (double)H;
    if ((y > dH && ye > dH) || (y < 0.0 && ye < 0.0) || (x > dW && xe > dW) || (x < 0.0 && xe < 0.0)) return;
    if (x > xe) { double t = x; x = xe; xe = t; t = y; y = ye; ye = t; }
    if (floor(x) == floor(xe) || fabs(dsub(x, xe)) < 0.01) {         // vertical
        if (ye < y) { const double t = y; y = ye; ye = t; }
        const int ix = (int)floor(xe);
        int iy = (int)floor(y), iye = (int)floor(ye);
        if (ix < 0 || ix >= W) return;
        iy = max(iy, 0);
        iye = min(iye, H - 1);
        for (; iy <= iye; iy++) burn(owner, W, iy, ix, f);
        return;
    }
    if (floor(y) == floor(ye) || fabs(dsub(y, ye)) < 0.01) {         // horizontal
        int ix = (int)floor(x);
        const int iy = (int)floor(y);
        int ixe = (int)floor(xe);
        if (iy < 0 || iy >= H) return;
        ix = max(ix, 0);
        ixe = min(ixe, W - 1);
        for (; ix <= ixe; ix++) burn(owner, W, iy, ix, f);
        return;
    }
    const double slope = ddiv(dsub(ye, y), dsub(xe, x));
    if (xe > dW) { ye = dsub(ye, dmul(dsub(xe, dW), slope)); xe = dW; }
    if (x < 0.0) { y = dadd(y, dmul(dsub(0.0, x), slope)); x = 0.0; }
    if (ye > y) {
        if (y < 0.0) { x = dadd(x, ddiv(dsub(0.0, y), slope)); y = 0.0; }
        if (ye >= dH) xe = dadd(xe, ddiv(dsub(ye, dH), slope));
    } else {
        if (y >= dH) { x = dadd(x, ddiv(dsub(dH, y), slope)); y = dH; }
        if (ye < 0.0) xe = dsub(xe, ddiv(dsub(ye, 0.0), slope));
    }
    while (x >= 0.0 && x < xe) {
        const int ix = (int)floor(x), iy = (int)floor(y);
        if (iy >= 0 && iy < H && ix < W) burn(owner, W, iy, ix, f);
        double step_x = dsub(floor(dadd(x, 1.0)), x);
        double step_y = dmul(step_x, slope);
        if ((int)floor(dadd(y, step_y)) == iy) {
            x = dadd(x, step_x);
            y = dadd(y, step_y);
        } else if (slope < 0) {
            step_y = dsub((double)iy, y);
            if (step_y > -0.000000001) step_y = -0.000000001;
            step_x = ddiv(step_y, slope);
            x = dadd(x, step_x);
            y = dadd(y, step_y);
        } else {
            step_y = dsub((double)(iy + 1), y);
            if (step_y < 0.000000001) step_y = 0.000000001;
            step_x = ddiv(step_y, slope);
            x = dadd(x, step_x);
            y = dadd(y, step_y);
        }
    }
}

// ---------------------------------------------------------------- label layer CRS -> tile CRS (WGS84 transverse Mercator)
// RasterizeLayer transforms every geometry from the layer's SRS to the raster's before it burns (OGR's on-the-fly
// reprojection, _descartes_img_chips.py:667-688); for label layers in longitude / latitude (EPSG:4326) or another UTM zone
// that is PROJ's `utm`: the Krueger series of order 6 in the third flattening n (Karney 2011, PROJ's default tmerc).
// Forward: conformal latitude, Gauss-Schreiber (xi', eta'), then xi + i eta = zeta' + sum_j alpha_j sin(2j zeta');
// inverse: zeta' = zeta - sum_j beta_j sin(2j zeta), Gauss-Schreiber back, Newton for tan(phi).  All IEEE double.
struct TmParams {
    double k0A;               // k0 * rectifying radius
    double e, e2m;            // eccentricity, 1 - e^2
    double alpha[6], beta[6];
};

// sum_{j=1..6} c_j sin(2j zeta), zeta = xi + i eta, by the complex Clenshaw recurrence: one sincos / sinh / cosh of
// (2 xi, 2 eta) per point.  b_k = c_k + 2 cos(2 zeta) b_{k+1} - b_{k+2};  sum = b_1 sin(2 zeta).
__device__ __forceinline__ double2 tm_sum(const double (&c)[6], double xi, double eta) {
    double s2, c2;
    sincos(2.0 * xi, &s2, &c2);
    const double sh2 = sinh(2.0 * eta), ch2 = cosh(2.0 * eta);
    const double ar = 2.0 * c2 * ch2, ai = -2.0 * s2 * sh2;        // 2 cos(2 zeta)
    double b1r = 0.0, b1i = 0.0, b2r = 0.0, b2i = 0.0;
#pragma unroll
    for (int k = 5; k >= 0; k--) {
        const double tr = ar * b1r - ai * b1i - b2r + c[k];
        const double ti = ar * b1i + ai * b1r - b2i;
        b2r = b1r; b2i = b1i; b1r = tr; b1i = ti;
    }
    const double sr = s2 * ch2, si = c2 * sh2;                     // sin(2 zeta)
    return make_double2(b1r * sr - b1i * si, b1r * si + b1i * sr);
}

// tan of the conformal latitude from tau = tan(phi): sinh(atanh(sin phi) - e atanh(e sin phi)) expanded with the
// subtraction rule of sinh, so that it stays accurate next to the poles (Karney 2011, eq. 7-9).
__device__ __forceinline__ double tm_taup(double tau, const TmParams& p) {
    const double sig = sinh(p.e * atanh(p.e * tau / hypot(1.0, tau)));
    return tau * hypot(1.0, sig) - sig * hypot(1.0, tau);
}

// (tau = tan(phi), longitude from the central meridian in degrees) -> (easting - 500 000, northing without false northing)
__device__ __forceinline__ double2 tm_forward(double tau, double dlam_deg, const TmParams& p) {
    double sl, cl;
    sincospi(dlam_deg / 180.0, &sl, &cl);
    const double taup = tm_taup(tau, p);
    const double xip = atan2(taup, cl), etap = asinh(sl / hypot(taup, cl));
    const double2 d = tm_sum(p.alpha, xip, etap);
    return make_double2(p.k0A * (etap + d.y), p.k0A * (xip + d.x));
}

// (easting - 500 000, northing without false northing) -> (tau = tan(phi), longitude from the central meridian in degrees)
__device__ __forceinline__ double2 tm_inverse(double x, double y, const TmParams& p) {
    const double xi = y / p.k0A, eta = x / p.k0A;
    const double2 d = tm_sum(p.beta, xi, eta);
    const double xip = xi - d.x, etap = eta - d.y;
    double s, c;
    sincos(xip, &s, &c);
    const double sh = sinh(etap);
    const double taup = s / hypot(sh, c);
    double tau = taup / p.e2m;                                     // within e^4 of the root: three Newton steps suffice
#pragma unroll
    for (int it = 0; it < 3; it++) {
        const double ta = tm_taup(tau, p);
        tau += (taup - ta) * (1.0 + p.e2m * tau * tau) / (p.e2m * hypot(1.0, tau) * hypot(1.0, ta));
    }
    return make_double2(tau, atan2(sh, c) * (180.0 / CUDART_PI));
}

// degrees -> [-180, 180); fmod is exact
__device__ __forceinline__ double wrap180(double d) {
    d = fmod(d, 360.0);
    return d >= 180.0 ? d - 360.0 : (d < -180.0 ? d + 360.0 : d);
}

// central meridian of a UTM zone; 0 for EPSG:4326 (zone 0)
__device__ __forceinline__ double meridian(int zone) { return zone ? (double)(6 * zone - 183) : 0.0; }

// One vertex.  zone 0 = EPSG:4326 (x = longitude, y = latitude, degrees); 1..60 = UTM zone with false northing fn.  A vertex
// the series is not valid for (non-finite, |lat| > 90, 90 degrees or more from the destination's central meridian) becomes
// (NaN, NaN): it cannot lie on a tile of that zone.
__device__ __forceinline__ double2 project_one(double2 v, int src_zone, double src_fn, int dst_zone, double dst_fn,
                                               const TmParams& p) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (!isfinite(v.x) || !isfinite(v.y)) return make_double2(nan, nan);
    double tau, dlam;                                              // tan(latitude); degrees east of dst's meridian
    if (src_zone == 0) {
        if (fabs(v.y) > 90.0) return make_double2(nan, nan);
        double s, c;
        sincos(v.y * (CUDART_PI / 180.0), &s, &c);                 // at +-90 degrees c is tiny, not 0: tau stays finite
        tau = s / c;
        dlam = wrap180(v.x - meridian(dst_zone));
    } else {
        const double2 t = tm_inverse(v.x - 500000.0, v.y - src_fn, p);
        tau = t.x;
        dlam = wrap180(t.y + (meridian(src_zone) - meridian(dst_zone)));
    }
    if (dst_zone == 0) return make_double2(dlam, atan(tau) * (180.0 / CUDART_PI));
    if (!(fabs(dlam) < 90.0)) return make_double2(nan, nan);
    const double2 xy = tm_forward(tau, dlam, p);
    return make_double2(xy.x + 500000.0, xy.y + dst_fn);
}

__global__ void __launch_bounds__(256)
project_points_kernel(const double2* __restrict__ in, double2* __restrict__ out, uint64_t n, int src_zone, double src_fn,
                      int dst_zone, double dst_fn, TmParams p) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        out[i] = project_one(in[i], src_zone, src_fn, dst_zone, dst_fn, p);
}

// EPSG code -> (zone, false northing); zone 0 = 4326, -1 = unsupported
int utm_zone_of(int epsg, double* fn) {
    *fn = 0.0;
    if (epsg == 4326) return 0;
    const int z = epsg % 100;
    if ((epsg / 100 != 326 && epsg / 100 != 327) || z < 1 || z > 60) return -1;
    if (epsg / 100 == 327) *fn = 10000000.0;
    return z;
}

// WGS84, k0 = 0.9996: the series coefficients from n (Karney 2011, eq. 14, 35, 36)
TmParams utm_params() {
    const double f = 1.0 / 298.257223563, a = 6378137.0, n = f / (2.0 - f);
    const double n2 = n * n, n3 = n2 * n, n4 = n3 * n, n5 = n4 * n, n6 = n5 * n;
    TmParams p;
    p.k0A = 0.9996 * a / (1.0 + n) * (1.0 + n2 / 4.0 + n4 / 64.0 + n6 / 256.0);
    p.e = sqrt(f * (2.0 - f));
    p.e2m = 1.0 - f * (2.0 - f);
    p.alpha[0] = n / 2.0 - 2.0 / 3.0 * n2 + 5.0 / 16.0 * n3 + 41.0 / 180.0 * n4 - 127.0 / 288.0 * n5 + 7891.0 / 37800.0 * n6;
    p.alpha[1] = 13.0 / 48.0 * n2 - 3.0 / 5.0 * n3 + 557.0 / 1440.0 * n4 + 281.0 / 630.0 * n5 - 1983433.0 / 1935360.0 * n6;
    p.alpha[2] = 61.0 / 240.0 * n3 - 103.0 / 140.0 * n4 + 15061.0 / 26880.0 * n5 + 167603.0 / 181440.0 * n6;
    p.alpha[3] = 49561.0 / 161280.0 * n4 - 179.0 / 168.0 * n5 + 6601661.0 / 7257600.0 * n6;
    p.alpha[4] = 34729.0 / 80640.0 * n5 - 3418889.0 / 1995840.0 * n6;
    p.alpha[5] = 212378941.0 / 319334400.0 * n6;
    p.beta[0] = n / 2.0 - 2.0 / 3.0 * n2 + 37.0 / 96.0 * n3 - 1.0 / 360.0 * n4 - 81.0 / 512.0 * n5 + 96199.0 / 604800.0 * n6;
    p.beta[1] = 1.0 / 48.0 * n2 + 1.0 / 15.0 * n3 - 437.0 / 1440.0 * n4 + 46.0 / 105.0 * n5 - 1118711.0 / 3870720.0 * n6;
    p.beta[2] = 17.0 / 480.0 * n3 - 37.0 / 840.0 * n4 - 209.0 / 4480.0 * n5 + 5569.0 / 90720.0 * n6;
    p.beta[3] = 4397.0 / 161280.0 * n4 - 11.0 / 504.0 * n5 - 830251.0 / 7257600.0 * n6;
    p.beta[4] = 4583.0 / 161280.0 * n5 - 108847.0 / 3991680.0 * n6;
    p.beta[5] = 20648693.0 / 638668800.0 * n6;
    return p;
}

__global__ void raster_init_kernel(int32_t* owner, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) owner[i] = -1;
}

__global__ void raster_finish_kernel(const int32_t* __restrict__ owner, const uint8_t* __restrict__ values, uint8_t background,
                                     uint8_t* __restrict__ out, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int32_t f = owner[i];
        out[i] = f < 0 ? background : values[f];
    }
}

}  // namespace
}  // namespace b2

using namespace b2;

extern "C" int b2_rasterize_polygons(b2_ctx* ctx, const double* fill_segs, const uint32_t* fill_seg_off, const int32_t* feat_miny,
                                     const uint32_t* job_off, uint32_t n_jobs, const double* line_segs, const uint32_t* line_seg_feat,
                                     uint32_t n_line_segs, const uint8_t* values, int n_features, int width, int height,
                                     int background, const uint64_t* job_ints_off, int32_t* owner_ws, int32_t* ints_ws, uint8_t* out,
                                     b2_stream stream) {
    B2_REQUIRE(ctx && out && owner_ws, "b2_rasterize_polygons: NULL argument");
    B2_REQUIRE(width > 0 && height > 0 && (uint64_t)width * height < (1ull << 31), "b2_rasterize_polygons: bad raster size");
    B2_REQUIRE(n_features >= 0 && background >= 0 && background <= 255, "b2_rasterize_polygons: bad argument");
    B2_REQUIRE(n_features == 0 || (fill_seg_off && feat_miny && job_off && values), "b2_rasterize_polygons: NULL feature table");
    B2_REQUIRE(n_jobs == 0 || (fill_segs && job_ints_off && ints_ws), "b2_rasterize_polygons: NULL fill table");
    B2_REQUIRE(n_line_segs == 0 || (line_segs && line_seg_feat), "b2_rasterize_polygons: NULL line table");
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t npix = (size_t)width * height;
    const unsigned gx = (unsigned)std::min<size_t>((npix + 255) / 256, (size_t)ctx->sm_count * 8);
    raster_init_kernel<<<gx, 256, 0, s>>>(owner_ws, npix);
    ctx->launches++;
    if (n_jobs) {
        raster_fill_kernel<<<(n_jobs + 127) / 128, 128, 0, s>>>(reinterpret_cast<const double4*>(fill_segs), fill_seg_off, feat_miny,
                                                                  job_off, n_features, n_jobs, width, height, job_ints_off, ints_ws,
                                                                  owner_ws);
        ctx->launches++;
    }
    if (n_line_segs) {
        raster_lines_kernel<<<(n_line_segs + 127) / 128, 128, 0, s>>>(reinterpret_cast<const double4*>(line_segs), line_seg_feat,
                                                                        n_line_segs, width, height, owner_ws);
        ctx->launches++;
    }
    raster_finish_kernel<<<gx, 256, 0, s>>>(owner_ws, values, (uint8_t)background, out, npix);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int b2_project_points(b2_ctx* ctx, const double* in_dev, double* out_dev, uint64_t n, int src_epsg, int dst_epsg,
                                 b2_stream stream) {
    double src_fn, dst_fn;
    const int src_zone = utm_zone_of(src_epsg, &src_fn), dst_zone = utm_zone_of(dst_epsg, &dst_fn);
    B2_REQUIRE(src_zone >= 0, "b2_project_points: unsupported source CRS EPSG:" + std::to_string(src_epsg) +
                                  " (EPSG:4326, 32601-32660 and 32701-32760 are supported)");
    B2_REQUIRE(dst_zone >= 0, "b2_project_points: unsupported destination CRS EPSG:" + std::to_string(dst_epsg) +
                                  " (EPSG:4326, 32601-32660 and 32701-32760 are supported)");
    B2_REQUIRE(ctx && (n == 0 || (in_dev && out_dev)), "b2_project_points: NULL argument");
    if (n == 0) return 0;
    DeviceGuard g(ctx->device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (src_epsg == dst_epsg) {
        if (in_dev != out_dev) B2_CUDA(cudaMemcpyAsync(out_dev, in_dev, n * sizeof(double2), cudaMemcpyDeviceToDevice, s));
        return 0;
    }
    static const TmParams params = utm_params();
    const unsigned gx = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 16);
    project_points_kernel<<<gx, 256, 0, s>>>(reinterpret_cast<const double2*>(in_dev), reinterpret_cast<double2*>(out_dev), n,
                                             src_zone, src_fn, dst_zone, dst_fn, params);
    ctx->launches++;
    B2_CUDA(cudaGetLastError());
    return 0;
}
