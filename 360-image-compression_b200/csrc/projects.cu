// MultiProject: the 14 rectilinear viewports of an ERP image used for the viewport PSNR / SSIM of `--test` and for the
// distortion loss of training (SURVEY.md s8f-2).  Replaces /root/reference/extension/projects_cuda.cu (init :7-126, update
// :127-136, forward :181-252, backward :257-329) and projects.hpp.
//
// Geometry (same expressions, same float/double promotions as the reference so that the sampling coordinates -- and with them
// the integer source pixels -- come out the same):
//   ray of viewport pixel (h, w):  (1, (w - cx) * w_stride, -(h - cy) * h_stride) normalised            projects_cuda.cu:7-19
//   rotation of viewport v:        R = Rod(-phi_v * column 1 of Rz) * Rz,  Rz = Rod((0, 0, theta_v))      :20-50, :99-121
//   ERP coordinate:                x = theta / pi * hx + hx,  y = -2 lat / pi * hy + hy                   :51-68
// Forward is a gather (HBM/L2-bound): one thread owns a viewport pixel, computes its four source offsets and weights once
// and walks the N*C planes; the 14 * h * w outputs of a plane are written coalesced.  The reference recomputes the floor /
// modulo / weights per output element.  Backward scatters with fp32 atomics like the reference (:274-298).
#include <algorithm>
#include <cmath>
#include "common.cuh"

namespace lic360 {

constexpr int kViews = 14;

// Rodrigues rotation matrices of 14 axis-angle vectors, host side, float arithmetic exactly as projects_mrod (:20-50)
static void rodrigues14(const float* x, const float* y, const float* z, float* data) {
    for (int i = 0; i < kViews; i++) {
        const int base = i * 9;
        for (int k = 0; k < 9; k++) data[base + k] = 0.f;
        const float norm = std::sqrt(x[i] * x[i] + y[i] * y[i] + z[i] * z[i]);
        if (norm == 0) {
            data[base] = 1.f; data[base + 4] = 1.f; data[base + 8] = 1.f;
            continue;
        }
        const float tx = x[i] / norm, ty = y[i] / norm, tz = z[i] / norm;
        const float c = std::cos(norm), s = std::sin(norm);
        data[base + 0] = c + (1 - c) * tx * tx;
        data[base + 1] = (1 - c) * tx * ty - s * tz;
        data[base + 2] = (1 - c) * tx * tz + s * ty;
        data[base + 3] = (1 - c) * ty * tx + s * tz;
        data[base + 4] = c + (1 - c) * ty * ty;
        data[base + 5] = (1 - c) * ty * tz - s * tx;
        data[base + 6] = (1 - c) * tz * tx - s * ty;
        data[base + 7] = (1 - c) * tz * ty + s * tx;
        data[base + 8] = c + (1 - c) * tz * tz;
    }
}

struct Rot14 { float r[kViews * 9]; };

// rays of all viewports: xyz[v][ps][3] = R_v * normalised ray (projects_init_xyz_kernel + gmm_kernel + gmm_transpose_kernel fused;
// R_v = r2_v * r1_v is evaluated with the running-sum order of gmm_kernel :69-83)
__global__ void projects_rays_kernel(float* __restrict__ xyz, const __grid_constant__ Rot14 r1, const __grid_constant__ Rot14 r2,
                                     int h_out, int w_out, float w_stride, float h_stride, float c_x, float c_y) {
    const int inner = h_out * w_out, total = kViews * inner;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int v = i / inner, ps = i % inner;
        const int w = ps % w_out, h = ps / w_out;
        const float x = 1.f;
        const float y = (w - c_x) * w_stride;
        const float z = (h - c_y) * h_stride;
        const float r = sqrtf(x * x + y * y + z * z);
        const float xa = x / r, xb = y / r, xc = -z / r;
        float R[9];
#pragma unroll
        for (int m = 0; m < 3; m++)
#pragma unroll
            for (int n = 0; n < 3; n++) {
                float sum = 0;
#pragma unroll
                for (int j = 0; j < 3; j++) sum += r2.r[v * 9 + m * 3 + j] * r1.r[v * 9 + j * 3 + n];
                R[m * 3 + n] = sum;
            }
        xyz[(size_t)i * 3 + 0] = xa * R[0] + xb * R[1] + xc * R[2];
        xyz[(size_t)i * 3 + 1] = xa * R[3] + xb * R[4] + xc * R[5];
        xyz[(size_t)i * 3 + 2] = xa * R[6] + xb * R[7] + xc * R[8];
    }
}

// projects_cal_xyz_kernel (:51-68): ray -> ERP sampling coordinate (x along the width, y along the height)
__global__ void projects_coords_kernel(const float* __restrict__ xyz, float* __restrict__ tf, int total, float hx, float hy, float pi) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const float lat = asinf(xyz[(size_t)i * 3 + 2]);
        const float tx = xyz[(size_t)i * 3], ty = xyz[(size_t)i * 3 + 1];
        float theta = atanf(ty / tx);
        if (tx <= 0) theta = ty > 0 ? theta + pi : theta - pi;
        tf[(size_t)i * 2] = theta / pi * hx + hx;
        tf[(size_t)i * 2 + 1] = -2 * lat / pi * hy + hy;
    }
}

struct Tap4 { int o00, o01, o10, o11; float w00, w01, w10, w11; };

// the four source pixels and bilinear weights of one viewport pixel (projects_forward_kernel :188-196)
__device__ __forceinline__ Tap4 bilinear_taps(float fx, float fy, int hs, int ws) {
    Tap4 t;
    const int tw = static_cast<int>(floorf(fx)), th = static_cast<int>(floorf(fy));
    const int pw = (tw + 1) % ws;
    const int ph = th + 1 >= hs ? hs - 1 : th + 1;
    const float tx = fx - tw, ty = fy - th;
    const float ntx = 1.f - tx, nty = 1.f - ty;
    t.o00 = th * ws + tw; t.o01 = th * ws + pw; t.o10 = ph * ws + tw; t.o11 = ph * ws + pw;
    t.w00 = ntx * nty; t.w01 = tx * nty; t.w10 = ntx * ty; t.w11 = tx * ty;
    return t;
}
__device__ __forceinline__ int nearest_tap(float fx, float fy, int hs, int ws) {  // :207-210, floor(double(x) + 0.5)
    const int tw = static_cast<int>(floor(fx + 0.5)) % ws;
    int th = static_cast<int>(floor(fy + 0.5));
    th = th >= hs ? hs - 1 : th;
    return th * ws + tw;
}

// out[(v * NC + plane) * inner + ps]; the reference's product order: in*ntx*nty + in*tx*nty + in*ntx*ty + in*tx*ty, left to right
template <bool NEAR>
__global__ void projects_forward_kernel(const float* __restrict__ in, const float* __restrict__ tf, float* __restrict__ out,
                                        int NC, int hs, int ws, int inner) {
    const int total = kViews * inner;
    const size_t plane = (size_t)hs * ws;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int v = i / inner, ps = i % inner;
        const float2 c = reinterpret_cast<const float2*>(tf)[i];
        float* o = out + ((size_t)v * NC) * inner + ps;
        if (NEAR) {
            const int off = nearest_tap(c.x, c.y, hs, ws);
            for (int p = 0; p < NC; p++) o[(size_t)p * inner] = __ldg(in + p * plane + off);
        } else {
            const int tw = static_cast<int>(floorf(c.x)), th = static_cast<int>(floorf(c.y));
            const int pw = (tw + 1) % ws;
            const int ph = th + 1 >= hs ? hs - 1 : th + 1;
            const float tx = c.x - tw, ty = c.y - th;
            const float ntx = 1.f - tx, nty = 1.f - ty;  // the reference's `1. - tx` is a double expression rounded to float: same value
            const int o00 = th * ws + tw, o01 = th * ws + pw, o10 = ph * ws + tw, o11 = ph * ws + pw;
            for (int p = 0; p < NC; p++) {
                const float* src = in + p * plane;
                o[(size_t)p * inner] = __ldg(src + o00) * ntx * nty + __ldg(src + o01) * tx * nty + __ldg(src + o10) * ntx * ty + __ldg(src + o11) * tx * ty;
            }
        }
    }
}

// scatter of the viewport gradients back onto the ERP grid + the accumulated weights (bottom_diff_[1]), :257-298
template <bool NEAR>
__global__ void projects_backward_kernel(const float* __restrict__ top, const float* __restrict__ tf, float* __restrict__ grad,
                                         float* __restrict__ count, int NC, int hs, int ws, int inner) {
    const int total = kViews * inner;
    const size_t plane = (size_t)hs * ws;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int v = i / inner, ps = i % inner;
        const float2 c = reinterpret_cast<const float2*>(tf)[i];
        const float* t = top + ((size_t)v * NC) * inner + ps;
        if (NEAR) {
            const int off = nearest_tap(c.x, c.y, hs, ws);
            for (int p = 0; p < NC; p++) {
                atomicAdd(grad + p * plane + off, t[(size_t)p * inner]);
                atomicAdd(count + p * plane + off, 1.f);
            }
        } else {
            const Tap4 k = bilinear_taps(c.x, c.y, hs, ws);
            for (int p = 0; p < NC; p++) {
                const float g = t[(size_t)p * inner];
                float* gp = grad + p * plane;
                float* cp = count + p * plane;
                atomicAdd(gp + k.o00, k.w00 * g); atomicAdd(cp + k.o00, k.w00);
                atomicAdd(gp + k.o01, k.w01 * g); atomicAdd(cp + k.o01, k.w01);
                atomicAdd(gp + k.o10, k.w10 * g); atomicAdd(cp + k.o10, k.w10);
                atomicAdd(gp + k.o11, k.w11 * g); atomicAdd(cp + k.o11, k.w11);
            }
        }
    }
}

// ---- view footprint: which cells of an h x w ERP grid a rectilinear view of any direction touches -------------------------------
// Cell (i, j) is the closed spherical rectangle of the grid points it is centred on, in ProjectsOp's convention (x = theta / pi * hx
// + hx, y = -2 lat / pi * hy + hy, hx = (w - 1) / 2, hy = (h - 1) / 2): x in [j - 1/2, j + 1/2] and y in [i - 1/2, i + 1/2], both
// clamped to the sphere, so columns 0 and w - 1 are the half cells on either side of the +-pi seam and rows 0 and h - 1 end in a
// pole.  A view's field is the closed frustum {d : |d.r| <= tan(a) d.f, |d.u| <= tan(a) d.f}: convex, inside one hemisphere, with
// four great-circle edges.  Two such closed regions meet iff a corner of one lies in the other or an edge of the field crosses an
// edge of the cell (a meridian arc, or a parallel: a small circle, crossed up to twice), so the predicate tests exactly that, in
// float64.  One thread per (view, cell); the work is h * w * V cells.
constexpr int kFootViews = 16;  // views per launch: their planes and corners travel in the kernel's parameters

struct FootViews {
    double nrm[kFootViews][4][3];  // inward normals of the four edge planes: tan(a) f -+ r, tan(a) f -+ u
    double cor[kFootViews][4][3];  // the four corners, unit vectors, in order round the field
};

struct Vec3 { double x, y, z; };
__device__ __forceinline__ Vec3 v3(const double* p) { return {p[0], p[1], p[2]}; }
__device__ __forceinline__ double dot3(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ Vec3 cross3(Vec3 a, Vec3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__device__ __forceinline__ Vec3 sph(double lon, double lat) { return {cos(lat) * cos(lon), cos(lat) * sin(lon), sin(lat)}; }

struct CellBox { double lc, hw, b0, b1; };  // longitude centre and half-width, latitude range [b0, b1]

__device__ __forceinline__ bool lon_in(double lon, const CellBox& c) { return fabs(remainder(lon - c.lc, 2 * M_PI)) <= c.hw; }

__device__ __forceinline__ bool in_cell(Vec3 p, const CellBox& c) {
    const double rho = hypot(p.x, p.y), lat = atan2(p.z, rho);
    if (lat < c.b0 || lat > c.b1) return false;
    return rho == 0 || lon_in(atan2(p.y, p.x), c);  // a pole lies on every meridian
}

__device__ __forceinline__ bool on_arc(Vec3 a, Vec3 b, Vec3 n, Vec3 p) {  // p on the great circle of a, b; the arc is shorter than pi
    return dot3(cross3(a, p), n) >= 0 && dot3(cross3(p, b), n) >= 0;
}

__device__ bool arc_meets_meridian(Vec3 a, Vec3 b, Vec3 n, double lon, const CellBox& c) {
    const Vec3 m = {-sin(lon), cos(lon), 0.0}, q = cross3(n, m);
    for (int s = 0; s < 2; s++) {
        const Vec3 p = s ? Vec3{-q.x, -q.y, -q.z} : q;
        if (p.x * cos(lon) + p.y * sin(lon) < 0) continue;  // the other half of the meridian's great circle
        const double lat = atan2(p.z, hypot(p.x, p.y));
        if (lat >= c.b0 && lat <= c.b1 && on_arc(a, b, n, p)) return true;
    }
    return false;
}

__device__ bool arc_meets_parallel(Vec3 a, Vec3 b, Vec3 n, double lat, const CellBox& c) {
    const double rho = hypot(n.x, n.y);
    if (rho == 0) return false;  // the equator's great circle: it meets a parallel nowhere or everywhere, and the meridians see it
    const double s = sin(lat), cl = cos(lat);
    const double along = -n.z * s / rho, disc = cl * cl - along * along;
    if (disc < 0) return false;
    const double hx = n.x / rho, hy = n.y / rho, perp = sqrt(disc);
    for (int k = 0; k < 2; k++) {
        const double t = k ? -perp : perp;
        const Vec3 p = {along * hx - t * hy, along * hy + t * hx, s};
        if (lon_in(atan2(p.y, p.x), c) && on_arc(a, b, n, p)) return true;
    }
    return false;
}

__global__ void view_footprint_kernel(const __grid_constant__ FootViews fv, int32_t* __restrict__ out, int h, int w) {
    const int v = blockIdx.y, cells = h * w;
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= cells) return;
    const int i = cell / w, j = cell % w;
    const double hx = (w - 1) / 2.0, hy = (h - 1) / 2.0;
    const double x0 = fmax(j - 0.5, 0.0), x1 = fmin(j + 0.5, w - 1.0);
    const double y0 = fmax(i - 0.5, 0.0), y1 = fmin(i + 0.5, h - 1.0);
    const double l0 = (x0 - hx) / hx * M_PI, l1 = (x1 - hx) / hx * M_PI;
    CellBox c;
    c.lc = 0.5 * (l0 + l1);
    c.hw = 0.5 * (l1 - l0);
    c.b1 = (hy - y0) / hy * M_PI_2;
    c.b0 = (hy - y1) / hy * M_PI_2;
    Vec3 nrm[4], cor[4];
#pragma unroll
    for (int k = 0; k < 4; k++) { nrm[k] = v3(fv.nrm[v][k]); cor[k] = v3(fv.cor[v][k]); }
    bool hit = false;
    for (int k = 0; k < 4 && !hit; k++) {  // a cell corner inside the field
        const Vec3 p = sph(k & 1 ? l1 : l0, k & 2 ? c.b1 : c.b0);
        hit = dot3(nrm[0], p) >= 0 && dot3(nrm[1], p) >= 0 && dot3(nrm[2], p) >= 0 && dot3(nrm[3], p) >= 0;
    }
    for (int k = 0; k < 4 && !hit; k++) hit = in_cell(cor[k], c);  // a field corner inside the cell
    for (int k = 0; k < 4 && !hit; k++) {  // a field edge across a cell edge
        const Vec3 a = cor[k], b = cor[(k + 1) & 3], n = cross3(a, b);
        for (int e = 0; e < 2 && !hit; e++) {
            const double lat = e ? c.b1 : c.b0;
            hit = arc_meets_meridian(a, b, n, e ? l1 : l0, c);
            if (!hit && fabs(lat) < M_PI_2) hit = arc_meets_parallel(a, b, n, lat, c);  // a pole is no edge
        }
    }
    out[(size_t)v * cells + cell] = hit ? 1 : 0;
}

// Rodrigues rotation of the axis-angle vector (x, y, z), float64; rodrigues14's expressions
static void rodrigues_f64(double x, double y, double z, double* R) {
    const double norm = std::sqrt(x * x + y * y + z * z);
    if (norm == 0) {
        for (int k = 0; k < 9; k++) R[k] = k % 4 == 0 ? 1.0 : 0.0;
        return;
    }
    const double tx = x / norm, ty = y / norm, tz = z / norm, c = std::cos(norm), s = std::sin(norm);
    R[0] = c + (1 - c) * tx * tx;      R[1] = (1 - c) * tx * ty - s * tz; R[2] = (1 - c) * tx * tz + s * ty;
    R[3] = (1 - c) * ty * tx + s * tz; R[4] = c + (1 - c) * ty * ty;      R[5] = (1 - c) * ty * tz - s * tx;
    R[6] = (1 - c) * tz * tx - s * ty; R[7] = (1 - c) * tz * ty + s * tx; R[8] = c + (1 - c) * tz * tz;
}

}  // namespace lic360

using namespace lic360;

extern "C" int lic360_view_footprint(int h, int w, int nviews, const float* theta_host, const float* phi_host, const float* fov_host,
                                     int32_t* out_dev, void* stream) {
    LIC360_CHECK_ARG(out_dev && theta_host && phi_host && fov_host && nviews > 0, "bad arguments");
    LIC360_CHECK_ARG(h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0, "h and w must be even and positive");
    LIC360_CHECK_ARG((size_t)nviews * h * w < (size_t)1 << 31, "output too large");
    for (int v = 0; v < nviews; v++) {
        LIC360_CHECK_ARG(std::isfinite(theta_host[v]) && std::isfinite(phi_host[v]), "view angles must be finite");
        LIC360_CHECK_ARG(fov_host[v] > 0 && fov_host[v] < 1, "fov must lie in (0, 1) (units of pi)");
    }
    const int threads = 128, cells = h * w;
    for (int v0 = 0; v0 < nviews; v0 += kFootViews) {
        const int nv = std::min(kFootViews, nviews - v0);
        FootViews fv;
        for (int v = 0; v < nv; v++) {
            // lic360_projects_init's rotation R = Rod(-phi * column 1 of Rz) * Rz, Rz = Rod((0, 0, theta)), here in float64
            const double th = (double)theta_host[v0 + v] * M_PI, ph = (double)phi_host[v0 + v] * M_PI;
            double r1[9], r2[9], R[9];
            rodrigues_f64(0, 0, th, r1);
            rodrigues_f64(r1[1] * -ph, r1[4] * -ph, r1[7] * -ph, r2);
            for (int m = 0; m < 3; m++)
                for (int n = 0; n < 3; n++) R[m * 3 + n] = r2[m * 3] * r1[n] + r2[m * 3 + 1] * r1[3 + n] + r2[m * 3 + 2] * r1[6 + n];
            const double ta = std::tan((double)fov_host[v0 + v] * M_PI / 2);
            const double f[3] = {R[0], R[3], R[6]}, r[3] = {R[1], R[4], R[7]}, u[3] = {R[2], R[5], R[8]};
            const double sr[4] = {-1, 1, 1, -1}, su[4] = {-1, -1, 1, 1};
            for (int k = 0; k < 4; k++) {
                double len = 0;
                for (int d = 0; d < 3; d++) {
                    const double e = k < 2 ? r[d] : u[d];
                    fv.nrm[v][k][d] = ta * f[d] + (k % 2 ? e : -e);
                    fv.cor[v][k][d] = f[d] + ta * (sr[k] * r[d] + su[k] * u[d]);
                    len += fv.cor[v][k][d] * fv.cor[v][k][d];
                }
                len = std::sqrt(len);
                for (int d = 0; d < 3; d++) fv.cor[v][k][d] /= len;
            }
        }
        const dim3 grid((cells + threads - 1) / threads, nv);
        view_footprint_kernel<<<grid, threads, 0, as_stream(stream)>>>(fv, out_dev + (size_t)v0 * cells, h, w);
        LAUNCH_CHECK();
    }
    return LIC360_OK;
}

extern "C" int lic360_projects_init(float* xyz_dev, int h_out, int w_out, const float* theta14, const float* phi14, float fov,
                                    void* stream) {
    LIC360_CHECK_ARG(xyz_dev && theta14 && phi14 && h_out > 1 && w_out > 1, "bad arguments");
    // projects.hpp:8-19 (angles arrive in units of pi) and projects_cuda.cu:84-121, host float arithmetic as written there
    const float pi = (float)std::acos(-1.0);
    float theta[kViews], phi[kViews];
    for (int i = 0; i < kViews; i++) { theta[i] = theta14[i] * pi; phi[i] = phi14[i] * pi; }
    const float fov_r = fov * pi;
    const float hfov = fov_r * h_out / w_out / 2;
    const float wfov = fov_r / 2;
    const float c_x = (float)((w_out - 1) / 2.0), c_y = (float)((h_out - 1) / 2.0);
    const float pi_2 = pi / 2;
    const float wangle = pi_2 - wfov, hangle = pi_2 - hfov;
    const float w_stride = 2 * std::sin(wfov) / std::sin(wangle) / (w_out - 1);
    const float h_stride = 2 * std::sin(hfov) / std::sin(hangle) / (h_out - 1);
    Rot14 r1, r2;
    float xa[kViews], ya[kViews], za[kViews];
    for (int i = 0; i < kViews; i++) { xa[i] = 0; ya[i] = 0; za[i] = theta[i]; }
    rodrigues14(xa, ya, za, r1.r);
    for (int i = 0; i < kViews; i++) {
        xa[i] = r1.r[i * 9 + 1] * (-phi[i]);
        ya[i] = r1.r[i * 9 + 4] * (-phi[i]);
        za[i] = r1.r[i * 9 + 7] * (-phi[i]);
    }
    rodrigues14(xa, ya, za, r2.r);
    const int total = kViews * h_out * w_out;
    projects_rays_kernel<<<stream_grid(total, 256), 256, 0, as_stream(stream)>>>(xyz_dev, r1, r2, h_out, w_out, w_stride, h_stride, c_x, c_y);
    LAUNCH_CHECK();
    return LIC360_OK;
}

extern "C" int lic360_projects_update(const float* xyz_dev, float* tf_dev, int h_out, int w_out, int H, int W, void* stream) {
    LIC360_CHECK_ARG(xyz_dev && tf_dev && h_out > 0 && w_out > 0 && H > 0 && W > 0, "bad arguments");
    const float pi = (float)std::acos(-1.0);
    const float hx = (float)((W - 1) / 2.0), hy = (float)((H - 1) / 2.0);
    const int total = kViews * h_out * w_out;
    projects_coords_kernel<<<stream_grid(total, 256), 256, 0, as_stream(stream)>>>(xyz_dev, tf_dev, total, hx, hy, pi);
    LAUNCH_CHECK();
    return LIC360_OK;
}

extern "C" int lic360_projects_forward(const float* in_dev, const float* tf_dev, float* out_dev, int NC, int H, int W, int h_out,
                                       int w_out, int nearest, void* stream) {
    LIC360_CHECK_ARG(in_dev && tf_dev && out_dev && NC > 0 && H > 0 && W > 0 && h_out > 0 && w_out > 0, "bad arguments");
    LIC360_CHECK_ARG((size_t)NC * H * W < (size_t)1 << 31, "input too large for 32-bit plane offsets");
    const int inner = h_out * w_out, total = kViews * inner;
    const int grid = stream_grid(total, 128);
    if (nearest) projects_forward_kernel<true><<<grid, 128, 0, as_stream(stream)>>>(in_dev, tf_dev, out_dev, NC, H, W, inner);
    else projects_forward_kernel<false><<<grid, 128, 0, as_stream(stream)>>>(in_dev, tf_dev, out_dev, NC, H, W, inner);
    LAUNCH_CHECK();
    return LIC360_OK;
}

extern "C" int lic360_projects_backward(const float* top_diff_dev, const float* tf_dev, float* bottom_diff_dev, float* count_dev,
                                        int NC, int H, int W, int h_out, int w_out, int nearest, void* stream) {
    LIC360_CHECK_ARG(top_diff_dev && tf_dev && bottom_diff_dev && count_dev && NC > 0 && H > 0 && W > 0, "bad arguments");
    LIC360_CHECK_ARG((size_t)NC * H * W < (size_t)1 << 31, "input too large for 32-bit plane offsets");
    const size_t bytes = (size_t)NC * H * W * sizeof(float);
    LIC360_CUDA(cudaMemsetAsync(bottom_diff_dev, 0, bytes, as_stream(stream)));  // caffe_gpu_set(..., 0, ...) :307-308, stream-ordered here
    LIC360_CUDA(cudaMemsetAsync(count_dev, 0, bytes, as_stream(stream)));
    const int inner = h_out * w_out, total = kViews * inner;
    const int grid = stream_grid(total, 128);
    if (nearest) projects_backward_kernel<true><<<grid, 128, 0, as_stream(stream)>>>(top_diff_dev, tf_dev, bottom_diff_dev, count_dev, NC, H, W, inner);
    else projects_backward_kernel<false><<<grid, 128, 0, as_stream(stream)>>>(top_diff_dev, tf_dev, bottom_diff_dev, count_dev, NC, H, W, inner);
    LAUNCH_CHECK();
    return LIC360_OK;
}
