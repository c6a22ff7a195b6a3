// Device-side forward kinematics + sphere / SDF verdict for the rollout cost kernel.
//
// This is the B200 replacement for robot_model::RobotModel::updateJointGroup + isStateValid, which the
// reference calls once per (rollout, timestep) from OptimizationTask::computeCollisionCost
// (reference src/planners/src/wrappers/stomp/OptimizationTask.cpp:183-204).
//
// Arithmetic contract (DESIGN.md "FK arithmetic"): every operation below is a single IEEE-754 binary64
// operation issued explicitly — fma() where a fused multiply-add is meant, a plain * or + otherwise —
// and this translation unit is compiled with -fmad=false so that ptxas neither fuses nor splits any of
// them.  A CPU that issues the same sequence gets bit-identical sphere centres, hence bit-identical
// collision verdicts.
#pragma once
// This header is also the one in-memory header of the run-time specialised state kernel (state_codegen.hpp hands
// its text to NVRTC with -DSTOMP_B200_NVRTC and the two capacity macros): no other include may be added below.
#ifdef STOMP_B200_NVRTC
typedef int int32_t;
typedef unsigned int uint32_t;
typedef unsigned char uint8_t;
typedef unsigned long long uint64_t;
typedef long long int64_t;
#else
#include <cstdint>

#include "../../include/stomp_b200.h"
#endif

namespace stomp_b200 {

enum AxisKind : int32_t { kAxisX = 0, kAxisY = 1, kAxisZ = 2, kAxisNegX = 3, kAxisNegY = 4, kAxisNegZ = 5, kAxisGeneral = 6 };

// one URDF joint, preprocessed on the host at stomp_b200_set_chain
struct JointParams {
    double o[3];      // origin xyz in the parent link frame
    double A[9];      // fixed rotation from rpy (row major)
    double axis[3];
    int32_t parent;   // -1: chain restarts at the base frame
    int32_t axis_kind;
    int32_t fixed_rot_identity;
    int32_t prismatic;
    int32_t o_mask;   // bit i set <=> o[i] != 0 (a zero component contributes fma(r, 0, p) == p: skipped)
    int32_t pad_;
};

struct SphereParams {
    double l[3];      // centre in the link frame
    double r;
    int32_t mask;     // bit i set <=> l[i] != 0
    float r_up;       // smallest binary32 >= r: for a binary32 distance d, (double)d - r < 0  <=>  d < r_up
};


// passed by value as a __grid_constant__ kernel parameter: lives in the constant bank, every access is
// warp-uniform
struct RobotParams {
    int32_t num_joints;
    int32_t num_spheres;
    int32_t simple_chain;     // every joint revolute, rpy == 0, axis along +-x / +-y / +-z (the usual URDF arm)
    int32_t pad_;
    int32_t sphere_begin[STOMP_B200_MAX_DIMS + 1];   // spheres of joint d: [sphere_begin[d], sphere_begin[d+1])
    double lower[STOMP_B200_MAX_DIMS];
    double upper[STOMP_B200_MAX_DIMS];
    JointParams joint[STOMP_B200_MAX_DIMS];
    SphereParams sphere[STOMP_B200_MAX_SPHERES];
};

struct SdfParams {
    const float* grid;
    int32_t nx, ny, nz;
    int32_t wide_index;        // 1 when nx*ny*nz does not fit 31 bits
    double offx, offy, offz;   // -(origin * inv_h)
    double inv_h;
};

// The field local query q reads: its record in the per-query table of an engine with several scenes, else the kernel's
// SdfParams argument.  The copy goes through a pointer to the chosen record: written as `table ? table[q] : arg` (or as a
// member-wise copy under an if) with a __grid_constant__ argument, nvcc 12.9 takes `grid` from the argument on both paths.
__device__ __forceinline__ SdfParams query_field(const SdfParams* table, int q, const SdfParams& arg)
{
    const SdfParams* src = table ? table + q : &arg;
    return *src;
}

// Deterministic sin/cos (also run on the host for the fixed rpy rotations of stomp_b200_set_chain, so
// that the whole FK is one arithmetic): 3-term Cody-Waite reduction by pi/2, then the degree-13 / degree-14 minimax
// polynomials on [-pi/4, pi/4] (coefficients of Sun's fdlibm kernels; mathematical constants).
// On the device the constants come from a __constant__ table: a constant-bank operand costs no instruction,
// while a 64-bit literal is materialised with two UMOVs every time the compiler runs out of uniform registers.
#define STOMP_B200_SINCOS_TABLE                                                                                  \
    6.36619772367581382433e-01, 1.57079632673412561417e+00, 6.07710050630396597660e-11, 2.02226624871116645580e-21, \
    1.58969099521155010221e-10, -2.50507602534068634195e-08, 2.75573137070700676789e-06, -1.98412698298579493134e-04, \
    8.33333333332248946124e-03, -1.66666666666666324348e-01, -1.13596475577881948265e-11, 2.08757232129817482790e-09, \
    -2.75573143513906633035e-07, 2.48015872894767294178e-05, -1.38888888888741095749e-03, 4.16666666666666019037e-02
__constant__ double kSinCosTable[16] = {STOMP_B200_SINCOS_TABLE};
#ifndef STOMP_B200_NVRTC
static const double kSinCosTableHost[16] = {STOMP_B200_SINCOS_TABLE};
#endif
#ifdef __CUDA_ARCH__
#define STOMP_B200_SC(i) kSinCosTable[i]
#else
#define STOMP_B200_SC(i) kSinCosTableHost[i]
#endif

__host__ __device__ __forceinline__ void det_sincos(double x, double& s_out, double& c_out)
{
    const double k = rint(x * STOMP_B200_SC(0));
    const double nk = -k;
    double r = fma(nk, STOMP_B200_SC(1), x);
    r = fma(nk, STOMP_B200_SC(2), r);
    r = fma(nk, STOMP_B200_SC(3), r);
    const double z = r * r;

    double ps = fma(z, STOMP_B200_SC(4), STOMP_B200_SC(5));
    ps = fma(z, ps, STOMP_B200_SC(6));
    ps = fma(z, ps, STOMP_B200_SC(7));
    ps = fma(z, ps, STOMP_B200_SC(8));
    ps = fma(z, ps, STOMP_B200_SC(9));
    const double rz = r * z;
    const double sr = fma(rz, ps, r);

    double pc = fma(z, STOMP_B200_SC(10), STOMP_B200_SC(11));
    pc = fma(z, pc, STOMP_B200_SC(12));
    pc = fma(z, pc, STOMP_B200_SC(13));
    pc = fma(z, pc, STOMP_B200_SC(14));
    pc = fma(z, pc, STOMP_B200_SC(15));
    const double zz = z * z;
    const double half = fma(z, -0.5, 1.0);
    const double cr = fma(zz, pc, half);

    const int q = (int)((long long)k & 3);
    const bool swap = q & 1;
    const double a = swap ? cr : sr;
    const double b = swap ? sr : cr;
    s_out = (q & 2) ? -a : a;
    // q: 0 -> c = cr ; 1 -> c = -sr ; 2 -> c = -cr ; 3 -> c = sr
    c_out = ((q == 1) || (q == 2)) ? -b : b;
}

struct Frame {
    double r00, r01, r02, r10, r11, r12, r20, r21, r22;
    double px, py, pz;
};

__device__ __forceinline__ void frame_identity(Frame& f)
{
    f.r00 = 1.0; f.r01 = 0.0; f.r02 = 0.0;
    f.r10 = 0.0; f.r11 = 1.0; f.r12 = 0.0;
    f.r20 = 0.0; f.r21 = 0.0; f.r22 = 1.0;
    f.px = 0.0; f.py = 0.0; f.pz = 0.0;
}

// rotate two columns (a, b) of the frame: a' = c*a + s*b ; b' = c*b - s*a   (row by row)
#define STOMP_B200_ROT2(a, b, s, ns, c)          \
    {                                            \
        const double _a = (a), _b = (b);         \
        (a) = fma((s), _b, (c) * _a);            \
        (b) = fma((ns), _a, (c) * _b);           \
    }

// kSimple: compiled without the fixed-rotation, prismatic and general-axis branches (RobotParams::simple_chain)
template <bool kSimple>
__device__ __forceinline__ void apply_joint(Frame& f, const JointParams& j, double q)
{
    if (j.parent < 0) frame_identity(f);
    // p += R * o, component by component in the order x, y, z; exact-zero components are skipped
    // (fma(r, 0, p) == p for finite r, so the result is the one the unskipped sequence gives)
    if (j.o_mask & 1) { f.px = fma(f.r00, j.o[0], f.px); f.py = fma(f.r10, j.o[0], f.py); f.pz = fma(f.r20, j.o[0], f.pz); }
    if (j.o_mask & 2) { f.px = fma(f.r01, j.o[1], f.px); f.py = fma(f.r11, j.o[1], f.py); f.pz = fma(f.r21, j.o[1], f.pz); }
    if (j.o_mask & 4) { f.px = fma(f.r02, j.o[2], f.px); f.py = fma(f.r12, j.o[2], f.py); f.pz = fma(f.r22, j.o[2], f.pz); }
    if (!kSimple && !j.fixed_rot_identity) {   // R = R * A
        const double n00 = fma(f.r02, j.A[6], fma(f.r01, j.A[3], f.r00 * j.A[0]));
        const double n01 = fma(f.r02, j.A[7], fma(f.r01, j.A[4], f.r00 * j.A[1]));
        const double n02 = fma(f.r02, j.A[8], fma(f.r01, j.A[5], f.r00 * j.A[2]));
        const double n10 = fma(f.r12, j.A[6], fma(f.r11, j.A[3], f.r10 * j.A[0]));
        const double n11 = fma(f.r12, j.A[7], fma(f.r11, j.A[4], f.r10 * j.A[1]));
        const double n12 = fma(f.r12, j.A[8], fma(f.r11, j.A[5], f.r10 * j.A[2]));
        const double n20 = fma(f.r22, j.A[6], fma(f.r21, j.A[3], f.r20 * j.A[0]));
        const double n21 = fma(f.r22, j.A[7], fma(f.r21, j.A[4], f.r20 * j.A[1]));
        const double n22 = fma(f.r22, j.A[8], fma(f.r21, j.A[5], f.r20 * j.A[2]));
        f.r00 = n00; f.r01 = n01; f.r02 = n02;
        f.r10 = n10; f.r11 = n11; f.r12 = n12;
        f.r20 = n20; f.r21 = n21; f.r22 = n22;
    }
    if (!kSimple && j.prismatic) {   // p += q * (R * axis)
        const double dx = fma(f.r02, j.axis[2], fma(f.r01, j.axis[1], f.r00 * j.axis[0]));
        const double dy = fma(f.r12, j.axis[2], fma(f.r11, j.axis[1], f.r10 * j.axis[0]));
        const double dz = fma(f.r22, j.axis[2], fma(f.r21, j.axis[1], f.r20 * j.axis[0]));
        f.px = fma(q, dx, f.px);
        f.py = fma(q, dy, f.py);
        f.pz = fma(q, dz, f.pz);
        return;
    }
    double s, c;
    det_sincos(q, s, c);
    int kind = j.axis_kind;
    if (kind >= kAxisNegX && kind <= kAxisNegZ) { s = -s; kind -= 3; }
    const double ns = -s;
    if (kind == kAxisZ) {          // col0' = c*col0 + s*col1 ; col1' = c*col1 - s*col0
        STOMP_B200_ROT2(f.r00, f.r01, s, ns, c)
        STOMP_B200_ROT2(f.r10, f.r11, s, ns, c)
        STOMP_B200_ROT2(f.r20, f.r21, s, ns, c)
    } else if (kind == kAxisY) {   // col0' = c*col0 - s*col2 ; col2' = c*col2 + s*col0
        STOMP_B200_ROT2(f.r00, f.r02, ns, s, c)
        STOMP_B200_ROT2(f.r10, f.r12, ns, s, c)
        STOMP_B200_ROT2(f.r20, f.r22, ns, s, c)
    } else if (kind == kAxisX) {   // col1' = c*col1 + s*col2 ; col2' = c*col2 - s*col1
        STOMP_B200_ROT2(f.r01, f.r02, s, ns, c)
        STOMP_B200_ROT2(f.r11, f.r12, s, ns, c)
        STOMP_B200_ROT2(f.r21, f.r22, s, ns, c)
    } else if (!kSimple) {         // Rodrigues: Q = c*I + s*[a]x + (1-c)*a a^T ; R = R*Q
        const double ax = j.axis[0], ay = j.axis[1], az = j.axis[2];
        const double v = 1.0 - c;
        const double vx = v * ax, vy = v * ay, vz = v * az;
        const double q00 = fma(vx, ax, c),          q01 = fma(vx, ay, -(s * az)), q02 = fma(vx, az, s * ay);
        const double q10 = fma(vy, ax, s * az),     q11 = fma(vy, ay, c),         q12 = fma(vy, az, -(s * ax));
        const double q20 = fma(vz, ax, -(s * ay)),  q21 = fma(vz, ay, s * ax),    q22 = fma(vz, az, c);
        const double n00 = fma(f.r02, q20, fma(f.r01, q10, f.r00 * q00));
        const double n01 = fma(f.r02, q21, fma(f.r01, q11, f.r00 * q01));
        const double n02 = fma(f.r02, q22, fma(f.r01, q12, f.r00 * q02));
        const double n10 = fma(f.r12, q20, fma(f.r11, q10, f.r10 * q00));
        const double n11 = fma(f.r12, q21, fma(f.r11, q11, f.r10 * q01));
        const double n12 = fma(f.r12, q22, fma(f.r11, q12, f.r10 * q02));
        const double n20 = fma(f.r22, q20, fma(f.r21, q10, f.r20 * q00));
        const double n21 = fma(f.r22, q21, fma(f.r21, q11, f.r20 * q01));
        const double n22 = fma(f.r22, q22, fma(f.r21, q12, f.r20 * q02));
        f.r00 = n00; f.r01 = n01; f.r02 = n02;
        f.r10 = n10; f.r11 = n11; f.r12 = n12;
        f.r20 = n20; f.r21 = n21; f.r22 = n22;
    }
}

__device__ __forceinline__ void sphere_centre(const Frame& f, const SphereParams& sp, double& cx, double& cy, double& cz)
{
    cx = f.px; cy = f.py; cz = f.pz;
    if (sp.mask & 1) { cx = fma(f.r00, sp.l[0], cx); cy = fma(f.r10, sp.l[0], cy); cz = fma(f.r20, sp.l[0], cz); }
    if (sp.mask & 2) { cx = fma(f.r01, sp.l[1], cx); cy = fma(f.r11, sp.l[1], cy); cz = fma(f.r21, sp.l[1], cz); }
    if (sp.mask & 4) { cx = fma(f.r02, sp.l[2], cx); cy = fma(f.r12, sp.l[2], cy); cz = fma(f.r22, sp.l[2], cz); }
}

// nearest-voxel lookup: voxel coordinate f = c * (1/h) - origin/h (one fma), truncated and clamped to the
// grid.  cvt.rzi.s32.f64 saturates and maps NaN to 0, so clamping the integer equals clamping the double
// to [0, n-1] first (what the CPU statement of the same rule does).
__device__ __forceinline__ size_t sdf_index(const SdfParams& g, double cx, double cy, double cz)
{
    const int ix = min(max(__double2int_rz(fma(cx, g.inv_h, g.offx)), 0), g.nx - 1);
    const int iy = min(max(__double2int_rz(fma(cy, g.inv_h, g.offy)), 0), g.ny - 1);
    const int iz = min(max(__double2int_rz(fma(cz, g.inv_h, g.offz)), 0), g.nz - 1);
    if (g.wide_index) return ((size_t)iz * (size_t)g.ny + (size_t)iy) * (size_t)g.nx + (size_t)ix;
    return (size_t)(unsigned)((iz * g.ny + iy) * g.nx + ix);
}

// ---------------------------------------------------------------------------------------------------
// Compile-time structured variants for the run-time specialised state kernel (state_codegen.hpp): the same
// operations in the same order as apply_joint / sphere_centre / sdf_index above, with every structural
// decision (axis kind, zero masks, fixed rotation, prismatic, index width) a template
// argument, so that the instantiated code is straight-line and every constant a direct constant-bank operand.
// ---------------------------------------------------------------------------------------------------
// everything of a joint that comes before its rotation: origin, fixed rotation; for a prismatic joint also the translation
// along its axis (the joint is then complete).  A chain restart is the caller's: it materialises the identity frame first.
template <int kOMask, bool kFixedRot, bool kPrismatic>
__device__ __forceinline__ void place_joint_static(Frame& f, const JointParams& j, double q)
{
    if (kOMask & 1) { f.px = fma(f.r00, j.o[0], f.px); f.py = fma(f.r10, j.o[0], f.py); f.pz = fma(f.r20, j.o[0], f.pz); }
    if (kOMask & 2) { f.px = fma(f.r01, j.o[1], f.px); f.py = fma(f.r11, j.o[1], f.py); f.pz = fma(f.r21, j.o[1], f.pz); }
    if (kOMask & 4) { f.px = fma(f.r02, j.o[2], f.px); f.py = fma(f.r12, j.o[2], f.py); f.pz = fma(f.r22, j.o[2], f.pz); }
    if (kFixedRot) {   // R = R * A
        const double n00 = fma(f.r02, j.A[6], fma(f.r01, j.A[3], f.r00 * j.A[0]));
        const double n01 = fma(f.r02, j.A[7], fma(f.r01, j.A[4], f.r00 * j.A[1]));
        const double n02 = fma(f.r02, j.A[8], fma(f.r01, j.A[5], f.r00 * j.A[2]));
        const double n10 = fma(f.r12, j.A[6], fma(f.r11, j.A[3], f.r10 * j.A[0]));
        const double n11 = fma(f.r12, j.A[7], fma(f.r11, j.A[4], f.r10 * j.A[1]));
        const double n12 = fma(f.r12, j.A[8], fma(f.r11, j.A[5], f.r10 * j.A[2]));
        const double n20 = fma(f.r22, j.A[6], fma(f.r21, j.A[3], f.r20 * j.A[0]));
        const double n21 = fma(f.r22, j.A[7], fma(f.r21, j.A[4], f.r20 * j.A[1]));
        const double n22 = fma(f.r22, j.A[8], fma(f.r21, j.A[5], f.r20 * j.A[2]));
        f.r00 = n00; f.r01 = n01; f.r02 = n02;
        f.r10 = n10; f.r11 = n11; f.r12 = n12;
        f.r20 = n20; f.r21 = n21; f.r22 = n22;
    }
    if (kPrismatic) {   // p += q * (R * axis)
        const double dx = fma(f.r02, j.axis[2], fma(f.r01, j.axis[1], f.r00 * j.axis[0]));
        const double dy = fma(f.r12, j.axis[2], fma(f.r11, j.axis[1], f.r10 * j.axis[0]));
        const double dz = fma(f.r22, j.axis[2], fma(f.r21, j.axis[1], f.r20 * j.axis[0]));
        f.px = fma(q, dx, f.px);
        f.py = fma(q, dy, f.py);
        f.pz = fma(q, dz, f.pz);
    }
}

// the rotation of a revolute joint from the sine / cosine of its value (the tail of apply_joint); the generated kernel
// evaluates the sines and cosines itself, inside each joint or a batch of joints up front (state_codegen.hpp:
// StateKernelOptions::batch_sincos) — the same operations on the same operands either way
template <int kKind>
__device__ __forceinline__ void rotate_joint_static(Frame& f, const JointParams& j, double s, double c)
{
    if (kKind >= kAxisNegX && kKind <= kAxisNegZ) s = -s;
    constexpr int kind = (kKind >= kAxisNegX && kKind <= kAxisNegZ) ? kKind - 3 : kKind;
    const double ns = -s;
    if (kind == kAxisZ) {
        STOMP_B200_ROT2(f.r00, f.r01, s, ns, c)
        STOMP_B200_ROT2(f.r10, f.r11, s, ns, c)
        STOMP_B200_ROT2(f.r20, f.r21, s, ns, c)
    } else if (kind == kAxisY) {
        STOMP_B200_ROT2(f.r00, f.r02, ns, s, c)
        STOMP_B200_ROT2(f.r10, f.r12, ns, s, c)
        STOMP_B200_ROT2(f.r20, f.r22, ns, s, c)
    } else if (kind == kAxisX) {
        STOMP_B200_ROT2(f.r01, f.r02, s, ns, c)
        STOMP_B200_ROT2(f.r11, f.r12, s, ns, c)
        STOMP_B200_ROT2(f.r21, f.r22, s, ns, c)
    } else {
        const double ax = j.axis[0], ay = j.axis[1], az = j.axis[2];
        const double v = 1.0 - c;
        const double vx = v * ax, vy = v * ay, vz = v * az;
        const double q00 = fma(vx, ax, c),          q01 = fma(vx, ay, -(s * az)), q02 = fma(vx, az, s * ay);
        const double q10 = fma(vy, ax, s * az),     q11 = fma(vy, ay, c),         q12 = fma(vy, az, -(s * ax));
        const double q20 = fma(vz, ax, -(s * ay)),  q21 = fma(vz, ay, s * ax),    q22 = fma(vz, az, c);
        const double n00 = fma(f.r02, q20, fma(f.r01, q10, f.r00 * q00));
        const double n01 = fma(f.r02, q21, fma(f.r01, q11, f.r00 * q01));
        const double n02 = fma(f.r02, q22, fma(f.r01, q12, f.r00 * q02));
        const double n10 = fma(f.r12, q20, fma(f.r11, q10, f.r10 * q00));
        const double n11 = fma(f.r12, q21, fma(f.r11, q11, f.r10 * q01));
        const double n12 = fma(f.r12, q22, fma(f.r11, q12, f.r10 * q02));
        const double n20 = fma(f.r22, q20, fma(f.r21, q10, f.r20 * q00));
        const double n21 = fma(f.r22, q21, fma(f.r21, q11, f.r20 * q01));
        const double n22 = fma(f.r22, q22, fma(f.r21, q12, f.r20 * q02));
        f.r00 = n00; f.r01 = n01; f.r02 = n02;
        f.r10 = n10; f.r11 = n11; f.r12 = n12;
        f.r20 = n20; f.r21 = n21; f.r22 = n22;
    }
}

// address of the voxel under one sphere centre (the gather itself is issued by the caller, so that the
// generated kernel can batch the loads of a link)
// floor of a voxel coordinate |v| < 2^31 on the FP64 pipe: v + (2^52 + 2^51) rounded towards -inf leaves
// floor(v) in the low word.  After the clamp to [0, n-1] floor and truncation agree (both send (-1, 0) to 0), so
// this is the same index as sdf_index's cvt.rzi — without the conversion, which runs on the quarter-rate XU pipe
// and was the busiest pipe of the kernel (ncu, profiles/r1j).  Only instantiated when the host has bounded the
// reach of the chain (state_codegen.hpp: magic_floor_is_safe).
__device__ __forceinline__ int voxel_floor_magic(double v) { return __double2loint(__dadd_rd(v, 6755399441055744.0)); }

// address of the voxel under a sphere centre that the generated kernel has formed itself (state_codegen.hpp:
// FoldingEmitter::centre).  kInside: the host has proved that no sphere centre can leave the grid (state_codegen.hpp:
// reach_is_inside_grid), so the clamps — six VIMNMX per sphere, an eighth of the kernel's instructions — are identities
// and are left out.
template <bool kWide, bool kMagic, bool kInside>
__device__ __forceinline__ const float* voxel_of_centre(double cx, double cy, double cz, const SdfParams& g)
{
    const double vx = fma(cx, g.inv_h, g.offx), vy = fma(cy, g.inv_h, g.offy), vz = fma(cz, g.inv_h, g.offz);
    int ix = kMagic ? voxel_floor_magic(vx) : __double2int_rz(vx);
    int iy = kMagic ? voxel_floor_magic(vy) : __double2int_rz(vy);
    int iz = kMagic ? voxel_floor_magic(vz) : __double2int_rz(vz);
    if (!kInside) {
        ix = min(max(ix, 0), g.nx - 1);
        iy = min(max(iy, 0), g.ny - 1);
        iz = min(max(iz, 0), g.nz - 1);
    }
    if (kWide) return g.grid + (((size_t)iz * (size_t)g.ny + (size_t)iy) * (size_t)g.nx + (size_t)ix);
    return g.grid + (unsigned)((iz * g.ny + iy) * g.nx + ix);
}

// The state half of the noise-less rollout (Stomp::doNoiselessRollout, stomp/src/Stomp.cpp:253-272) and the wrapper's stop
// rule (src/wrappers/stomp/StompPlanner.cpp:107-118) as a TAIL of the state kernel: T extra states read from the padded
// policy rows, and the thread that finishes last — found with one packed atomic: hits in the low half, finished states in
// the high half — adds the control costs the update kernel left in the record, and does the bookkeeping.  theta == null:
// no tail.
struct NoiselessTail {
    const double* theta;           // [Q][D][N] + kPad: first free parameter of joint 0
    int32_t row_stride;            // N
    int32_t sumw;
    int64_t query_stride;          // D * N
    double* state;                 // [Q][T]   noiseless_rollout_.state_costs_
    uint8_t* verdict;              // [Q][T]
    uint8_t* valid;                // [Q]      last_noiseless_rollout_valid_
    double* sums;                  // [Q][sumw] the record: [0] <- S, [1 .. D] control-cost sums (already there)
    double* total;                 // [Q] noise-less total cost
    double* best;                  // [Q]
    double* old_cost;              // [Q]
    double* improvement;           // [Q]
    int32_t* iters;                // [Q]
    int32_t* stop;                 // [Q]
    uint32_t* counter;             // [Q] zero between launches
    int32_t* note;                 // [Q][2] host-mapped pinned words (iterations recorded, stopped) the host paces stomp_b200_solve by; may be null
    double min_cost_improvement;
};

// the sphere-pair rule (stomp_b200_set_self_collision): the list as the host sorted it
struct SelfPairs {
    const int2* ij;              // [n] sphere indices, x < y, sorted by (link of x, link of y)
    const double* limit2;        // [n] (r_x + r_y)^2
    const int4* block;           // [nblocks] (link a, link b, first pair, end pair)
    const double* block_limit2;  // [nblocks] (bound_a + bound_b)^2 of the inflated bounding radii
    const double* link_bound;    // [D][4] bounding sphere of a link's spheres in the link frame: x, y, z, (unused)
    int32_t n, nblocks;
};

// arguments of every state kernel (generated, generic, pair rule); filled only by the builders in engine.cu
struct StateKernelArgs {
    const double* rollouts;        // [Q][slots][D][T]
    double* state_costs;           // [Q][slots][T]
    uint8_t* verdicts;             // [Q][slots][T]
    uint8_t* validity;             // [Q][slots]
    double* sums;                  // [Q][gslots][sumw]
    double* s_compact;             // [Q][gslots] mirror of S_k for the fused weights + update kernel, or null
    const int32_t* stop;           // [Q]
    uint32_t* tile_counter;        // [4]
    unsigned long long* timeline;  // first-start / last-end stamps of this kernel, or null
    int32_t T, D, slots, gslots, sumw, num_gen, gen_offset, honour_stop;
    int32_t row_stride;            // doubles between consecutive joints of one rollout (T; N for the padded policy rows)
    int64_t rollout_stride;        // doubles between consecutive rollouts (D * T)
    NoiselessTail nl;
    // verdict of the spheres whose centres no joint value moves (state_codegen.hpp: FoldingEmitter::centre_is_static), written
    // once per robot / scene by stomp_b200_static_spheres; null when the kernel walks every sphere itself
    const int32_t* static_hit;
    // floor(2^32 / T) + 1 when num_gen * T * T < 2^32 (then umulhi(idx, t_magic) == idx / T for every state index), else 0
    uint32_t t_magic;
    // an engine with several scenes (stomp_b200_set_query_scenes): [Q] the field of each local query's scene and [Q] the
    // scene itself (static_hit then holds one verdict per scene).  Null: every query reads the SdfParams argument and
    // static_hit is that field's verdict
    const SdfParams* query_sdf;
    const int32_t* query_scene;
};

}  // namespace stomp_b200
