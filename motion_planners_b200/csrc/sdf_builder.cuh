// Environment -> signed distance field, on the device (SURVEY.md §8f rank 2).
//
// The reference keeps its world as collision objects handed to FCL — primitives, meshes and an octomap
// (src/MotionPlanners.cpp:162-173 assignOctomapPlanningScene / updateOctomap, :416-495 handleCollisionObjectInWorld /
// handleGraspObject, include/motion_planners/Config.hpp:14-35) — and asks FCL per state.  Here the world is a distance
// field the state kernel gathers from, so the world objects are turned into that field once per scene change:
//   * primitives (sphere / box): exact signed distance of the union at every voxel centre, one thread per voxel
//     (build_sdf_primitives_kernel);
//   * occupancy (a voxelised mesh or an octomap's leaf grid): exact Euclidean distance transform, three separable
//     min-plus passes over squared integer distances (edt_pass_kernel), signed by running it on the occupancy and on its
//     complement (finish_edt_kernel).
// Arithmetic contract (the oracle's oracle_build_sdf_* issue the same operations; bit-identical grids): FP64, one IEEE
// operation per source operation (-fmad=false), voxel centre = origin + (i + 0.5) * h, distances rounded to binary32.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace stomp_b200 {

constexpr int kMaxPrimitives = 256;

struct PrimitiveList {
    int32_t n;
    int32_t kind[kMaxPrimitives];        // 0 sphere (size[0] = radius), 1 box (size = half extents), 2 cylinder along z (radius, half height)
    double centre[kMaxPrimitives][3];
    double size[kMaxPrimitives][3];
};

// signed distance from p to one primitive (negative inside)
__device__ __forceinline__ double primitive_distance(int kind, const double* c, const double* s, double px, double py, double pz)
{
    const double dx = px - c[0], dy = py - c[1], dz = pz - c[2];
    if (kind == 0) return sqrt((dx * dx + dy * dy) + dz * dz) - s[0];
    if (kind == 2) {      // cylinder along z: s[0] radius, s[1] half height
        const double qr = sqrt(dx * dx + dy * dy) - s[0], qh = fabs(dz) - s[1];
        const double orr = fmax(qr, 0.0), oh = fmax(qh, 0.0);
        return sqrt(orr * orr + oh * oh) + fmin(fmax(qr, qh), 0.0);
    }
    const double qx = fabs(dx) - s[0], qy = fabs(dy) - s[1], qz = fabs(dz) - s[2];
    const double ox = fmax(qx, 0.0), oy = fmax(qy, 0.0), oz = fmax(qz, 0.0);
    const double outside = sqrt((ox * ox + oy * oy) + oz * oz);
    const double inside = fmin(fmax(fmax(qx, qy), qz), 0.0);
    return outside + inside;
}

// grid[(z * ny + y) * nx + x] = (float) min_i d_i(centre of voxel (x, y, z)); the list lives in global memory (one
// broadcast load per primitive and warp).  grid (ceil(nx / 128), ny, nz) — x along the thread index: coalesced stores.
__global__ void __launch_bounds__(128)
build_sdf_primitives_kernel(float* __restrict__ grid, int nx, int ny, int nz, double ox, double oy, double oz, double h,
                            const PrimitiveList* __restrict__ list)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y, z = blockIdx.z;
    if (x >= nx) return;
    const double px = ox + ((double)x + 0.5) * h, py = oy + ((double)y + 0.5) * h, pz = oz + ((double)z + 0.5) * h;
    double d = __longlong_as_double(0x7ff0000000000000ll);       // +inf
    const int n = list->n;
    for (int i = 0; i < n; ++i) d = fmin(d, primitive_distance(list->kind[i], list->centre[i], list->size[i], px, py, pz));
    grid[((size_t)z * ny + y) * nx + x] = (float)d;
}

// ---- exact Euclidean distance transform of an occupancy grid ---------------------------------------------------
// Squared distances in voxel units are integers: three passes of  out(i) = min_j (i - j)^2 + in(j)  along x, y, z
// (min-plus with a parabola; exact in int32 for grids up to 1024^3: 3 * 1023^2 < 2^31).  O(n) per voxel and pass — a
// 256^3 grid is 13 G integer operations, milliseconds on a B200, once per scene change; the O(1) lower-envelope sweep
// of Felzenszwalb & Huttenlocher is sequential along a line and does not map to a warp.
// One CTA per line: the line is staged in shared memory, thread i scans it.
constexpr int kEdtInf = 0x3fffffff;

__global__ void __launch_bounds__(256)
edt_pass_kernel(const int32_t* __restrict__ in, int32_t* __restrict__ out, int n_line, long long stride_line,
                int n_a, long long stride_a, long long stride_b)
{
    extern __shared__ int32_t line[];
    const size_t base = (size_t)blockIdx.x * stride_a + (size_t)blockIdx.y * stride_b;
    (void)n_a;
    for (int i = threadIdx.x; i < n_line; i += blockDim.x) line[i] = in[base + (size_t)i * stride_line];
    __syncthreads();
    for (int i = threadIdx.x; i < n_line; i += blockDim.x) {
        int best = kEdtInf;
        for (int j = 0; j < n_line; ++j) {
            const int v = line[j];
            const int dj = i - j;
            const int cand = (v >= kEdtInf) ? kEdtInf : v + dj * dj;
            best = min(best, cand);
        }
        out[base + (size_t)i * stride_line] = best;
    }
}

// seeds of the two transforms: distance to the nearest occupied voxel (0 on occupied voxels) and to the nearest free one
__global__ void edt_seed_kernel(const uint8_t* __restrict__ occupied, int32_t* __restrict__ to_occupied,
                                int32_t* __restrict__ to_free, size_t count)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const bool occ = occupied[i] != 0;
    to_occupied[i] = occ ? 0 : kEdtInf;
    to_free[i] = occ ? kEdtInf : 0;
}

// signed distance of the voxel centre to the occupied set's boundary voxels, in metres: +h * sqrt(d2 to the nearest
// occupied voxel) outside, -h * sqrt(d2 to the nearest free voxel) inside (centre-to-centre; a scene without occupied
// voxels is +inf-like: h * sqrt(kEdtInf))
__global__ void finish_edt_kernel(const uint8_t* __restrict__ occupied, const int32_t* __restrict__ to_occupied,
                                  const int32_t* __restrict__ to_free, float* __restrict__ grid, double h, size_t count)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const bool occ = occupied[i] != 0;
    const double d2 = (double)(occ ? to_free[i] : to_occupied[i]);
    const double d = h * sqrt(d2);
    grid[i] = (float)(occ ? -d : d);
}

// ---- meshes and octomap leaves -> occupancy ---------------------------------------------------------------------
// A triangle mesh (the reference's MESH model objects and the robot's own STL collision meshes, test/data/meshes/**) is
// voxelised conservatively: a voxel is occupied when its cube and a triangle overlap (separating-axis test of a box and a
// triangle: 3 box axes, the triangle's plane, 9 edge cross products), which makes the shell of a closed mesh 26-separating,
// so the interior can be found afterwards as the free voxels NOT reachable from the grid's boundary (6-connected flood,
// run as line sweeps until nothing changes).  An octomap arrives as its occupied leaves (centre + edge length): every
// voxel whose centre lies in a leaf's cube is occupied.  Arithmetic as everywhere in this file: FP64, one operation per
// source operation, restated by the oracle (oracle_build_sdf_scene) — identical occupancy, hence an identical field.
__device__ __forceinline__ bool triangle_overlaps_box(const double* tri /*[3][3]*/, double cx, double cy, double cz, double hh)
{
    const double v0x = tri[0] - cx, v0y = tri[1] - cy, v0z = tri[2] - cz;
    const double v1x = tri[3] - cx, v1y = tri[4] - cy, v1z = tri[5] - cz;
    const double v2x = tri[6] - cx, v2y = tri[7] - cy, v2z = tri[8] - cz;
    // box axes
    if (fmin(fmin(v0x, v1x), v2x) > hh || fmax(fmax(v0x, v1x), v2x) < -hh) return false;
    if (fmin(fmin(v0y, v1y), v2y) > hh || fmax(fmax(v0y, v1y), v2y) < -hh) return false;
    if (fmin(fmin(v0z, v1z), v2z) > hh || fmax(fmax(v0z, v1z), v2z) < -hh) return false;
    const double e0x = v1x - v0x, e0y = v1y - v0y, e0z = v1z - v0z;
    const double e1x = v2x - v1x, e1y = v2y - v1y, e1z = v2z - v1z;
    const double e2x = v0x - v2x, e2y = v0y - v2y, e2z = v0z - v2z;
    // triangle plane
    const double nx = e0y * e1z - e0z * e1y, ny = e0z * e1x - e0x * e1z, nz = e0x * e1y - e0y * e1x;
    const double dist = (nx * v0x + ny * v0y) + nz * v0z;
    const double rad = hh * ((fabs(nx) + fabs(ny)) + fabs(nz));
    if (dist > rad || dist < -rad) return false;
    // 9 edge x axis tests: axis a = e x unit_j; the triangle's projections onto a against the box's radius
#define STOMP_B200_AXIS(ax, ay, az)                                                                          \
    {                                                                                                        \
        const double p0 = ((ax) * v0x + (ay) * v0y) + (az) * v0z;                                            \
        const double p1 = ((ax) * v1x + (ay) * v1y) + (az) * v1z;                                            \
        const double p2 = ((ax) * v2x + (ay) * v2y) + (az) * v2z;                                            \
        const double r = hh * ((fabs(ax) + fabs(ay)) + fabs(az));                                            \
        if (fmin(fmin(p0, p1), p2) > r || fmax(fmax(p0, p1), p2) < -r) return false;                         \
    }
    STOMP_B200_AXIS(0.0, -e0z, e0y) STOMP_B200_AXIS(e0z, 0.0, -e0x) STOMP_B200_AXIS(-e0y, e0x, 0.0)
    STOMP_B200_AXIS(0.0, -e1z, e1y) STOMP_B200_AXIS(e1z, 0.0, -e1x) STOMP_B200_AXIS(-e1y, e1x, 0.0)
    STOMP_B200_AXIS(0.0, -e2z, e2y) STOMP_B200_AXIS(e2z, 0.0, -e2x) STOMP_B200_AXIS(-e2y, e2x, 0.0)
#undef STOMP_B200_AXIS
    return true;
}

// voxel index range [lo, hi] along one axis whose cubes can touch the interval [a, b] (clamped to the grid; empty if lo > hi)
__device__ __forceinline__ void voxel_range(double a, double b, double origin, double inv_h, int n, int& lo, int& hi)
{
    const double fa = floor((a - origin) * inv_h), fb = floor((b - origin) * inv_h);
    lo = (int)fmax(fa - 1.0, 0.0);
    hi = (int)fmin(fb + 1.0, (double)(n - 1));
    if (!(fb + 1.0 >= 0.0) || !(fa - 1.0 <= (double)(n - 1))) { lo = 1; hi = 0; }
}

// one CTA per triangle: the voxels of its bounding box (one voxel of slack) are tested by the CTA's threads
__global__ void __launch_bounds__(128)
voxelise_triangles_kernel(const double* __restrict__ triangles, int num_triangles, uint8_t* __restrict__ occ,
                          int nx, int ny, int nz, double ox, double oy, double oz, double h)
{
    const int tr = blockIdx.x;
    if (tr >= num_triangles) return;
    __shared__ double tri[9];
    if (threadIdx.x < 9) tri[threadIdx.x] = triangles[(size_t)tr * 9 + threadIdx.x];
    __syncthreads();
    // half edge of the test cube, inflated by 1e-9: a face lying exactly on a voxel boundary must not fall between the two
    // neighbouring cubes through rounding (it would open a hole in the shell and the interior fill would leak)
    const double inv_h = 1.0 / h, hh = (0.5 * h) * 1.000000001;
    int x0, x1, y0, y1, z0, z1;
    voxel_range(fmin(fmin(tri[0], tri[3]), tri[6]), fmax(fmax(tri[0], tri[3]), tri[6]), ox, inv_h, nx, x0, x1);
    voxel_range(fmin(fmin(tri[1], tri[4]), tri[7]), fmax(fmax(tri[1], tri[4]), tri[7]), oy, inv_h, ny, y0, y1);
    voxel_range(fmin(fmin(tri[2], tri[5]), tri[8]), fmax(fmax(tri[2], tri[5]), tri[8]), oz, inv_h, nz, z0, z1);
    if (x0 > x1 || y0 > y1 || z0 > z1) return;
    const int wx = x1 - x0 + 1, wy = y1 - y0 + 1, wz = z1 - z0 + 1;
    const long long total = (long long)wx * wy * wz;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
        const int x = x0 + (int)(i % wx), y = y0 + (int)((i / wx) % wy), z = z0 + (int)(i / ((long long)wx * wy));
        const double cx = ox + ((double)x + 0.5) * h, cy = oy + ((double)y + 0.5) * h, cz = oz + ((double)z + 0.5) * h;
        if (triangle_overlaps_box(tri, cx, cy, cz, hh)) occ[((size_t)z * ny + y) * nx + x] = 1;
    }
}

// octomap leaves: voxels whose centre lies in the leaf's cube [c - s/2, c + s/2]; one warp-sized CTA per leaf
__global__ void __launch_bounds__(32)
voxelise_leaves_kernel(const double* __restrict__ centres, const double* __restrict__ sizes, int num_leaves, uint8_t* __restrict__ occ,
                       int nx, int ny, int nz, double ox, double oy, double oz, double h)
{
    const int lf = blockIdx.x;
    if (lf >= num_leaves) return;
    const double inv_h = 1.0 / h, half = 0.5 * sizes[lf];
    int lo[3], hi[3];
    const double org[3] = {ox, oy, oz};
    const int nn[3] = {nx, ny, nz};
    for (int a = 0; a < 3; ++a) {
        const double c = centres[(size_t)lf * 3 + a];
        // centre of voxel i is origin + (i + 0.5) h: inside [c - half, c + half]  <=>  (c - half - origin) / h - 0.5 <= i <= (c + half - origin) / h - 0.5
        const double fl = ceil((c - half - org[a]) * inv_h - 0.5), fh = floor((c + half - org[a]) * inv_h - 0.5);
        lo[a] = (int)fmax(fl, 0.0);
        hi[a] = (int)fmin(fh, (double)(nn[a] - 1));
        if (!(fh >= 0.0) || !(fl <= (double)(nn[a] - 1))) return;
    }
    const int wx = hi[0] - lo[0] + 1, wy = hi[1] - lo[1] + 1, wz = hi[2] - lo[2] + 1;
    if (wx <= 0 || wy <= 0 || wz <= 0) return;
    const long long total = (long long)wx * wy * wz;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
        const int x = lo[0] + (int)(i % wx), y = lo[1] + (int)((i / wx) % wy), z = lo[2] + (int)(i / ((long long)wx * wy));
        occ[((size_t)z * ny + y) * nx + x] = 1;
    }
}

// interior of closed shells: `outside` = free voxels connected to the grid's boundary.  Seed, then line sweeps.
__global__ void flood_seed_kernel(const uint8_t* __restrict__ occ, uint8_t* __restrict__ outside, int nx, int ny, int nz)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t count = (size_t)nx * ny * nz;
    if (i >= count) return;
    const int x = (int)(i % nx), y = (int)((i / nx) % ny), z = (int)(i / ((size_t)nx * ny));
    const bool border = x == 0 || y == 0 || z == 0 || x == nx - 1 || y == ny - 1 || z == nz - 1;
    outside[i] = (border && !occ[i]) ? 1 : 0;
}
// one thread per line along an axis: forward and backward propagation of `outside` through free voxels
__global__ void flood_sweep_kernel(const uint8_t* __restrict__ occ, uint8_t* __restrict__ outside, int n_line, long long stride_line,
                                   int n_a, long long stride_a, int n_b, long long stride_b, int* __restrict__ changed)
{
    const long long l = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= (long long)n_a * n_b) return;
    const size_t base = (size_t)(l % n_a) * stride_a + (size_t)(l / n_a) * stride_b;
    bool any = false;
    bool prev = outside[base] != 0;
    for (int i = 1; i < n_line; ++i) {
        const size_t o = base + (size_t)i * stride_line;
        bool cur = outside[o] != 0;
        if (!cur && prev && !occ[o]) { outside[o] = 1; cur = true; any = true; }
        prev = cur;
    }
    prev = outside[base + (size_t)(n_line - 1) * stride_line] != 0;
    for (int i = n_line - 2; i >= 0; --i) {
        const size_t o = base + (size_t)i * stride_line;
        bool cur = outside[o] != 0;
        if (!cur && prev && !occ[o]) { outside[o] = 1; cur = true; any = true; }
        prev = cur;
    }
    if (any) *changed = 1;
}
__global__ void flood_fill_kernel(uint8_t* __restrict__ occ, const uint8_t* __restrict__ outside, size_t count)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count && !outside[i]) occ[i] = 1;
}

}  // namespace stomp_b200
