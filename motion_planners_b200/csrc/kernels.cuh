// sm_100a kernels of the STOMP rollout loop.  One translation unit (engine.cu) includes this file and is
// compiled with -fmad=false: fused multiply-adds appear only where fma() is written (kinematics.cuh
// states why).  Each kernel names the reference loop it replaces (SURVEY.md §2.1, K1-K11); paths are
// relative to /root/reference/src/planners/.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kinematics.cuh"

namespace stomp_b200 {

constexpr int kPad = 6;                 // TRAJECTORY_PADDING, stomp/include/stomp/StompUtils.hpp:57
constexpr int kMaxRules = 4;            // NUM_DIFF_RULES
constexpr int kRBand = 6;               // half bandwidth of R = sum D^T W D (7-tap rules)

// shape + pointers shared by every kernel (device memory; layouts in DESIGN.md "Data layout in HBM")
struct LoopParams {
    int32_t T, D, N, Q;
    int32_t slots;            // rollout slots per query in the local tensors (max_rollouts + 1)
    int32_t gslots;           // slots per query in the rollout-indexed scalar tables (global over ranks)
    int32_t sumw;             // 1 + 3*D doubles per rollout: S, C_d[D], cum_d[D], quad_d[D] (n^T R n)
    int32_t num_gen;          // G: rollouts generated this iteration (local)
    int32_t num_rollouts;     // K': rollouts used in the update (global over ranks)
    int32_t num_local;        // local rollout slots in use (generated + reused + noise-less)
    int32_t gen_offset;       // global index of local generated rollout 0 (rank * G)
    int32_t noiseless_slot;   // local slot of the appended noise-less rollout, -1 if none
    int32_t noiseless_gslot;  // its global slot
    int32_t honour_stop;
    int32_t iteration;
    int32_t store_control;    // write per-(k,d,t) control costs
    int32_t store_unit;       // write unit noise / epsilon (debug)
    int32_t use_noise_adaptation;
    int32_t query_offset;     // global index of local query 0
    int32_t gen_global;       // generated rollouts per query over all ranks (Philox column numbering)
    double control_cost_weight, dt, cost_scaling_h, min_cost_improvement;
    uint64_t seed;

    double* theta_all;        // [Q][D][N]
    const double* mincc;      // [Q][D][T]
    double* rollouts;         // [Q][slots][D][T]   parameters_noise_
    double* noise;            // [Q][slots][D][T]   noise_
    double* proj;             // [Q][slots][D][T]   parameters_noise_projected_ (reuse only) or null
    double* state_costs;      // [Q][slots][T]
    uint8_t* verdicts;        // [Q][slots][T]
    uint8_t* validity;        // [Q][slots]
    double* control_costs;    // [Q][slots][D][T] or null
    double* sums;             // [Q][gslots][sumw]
    double* total_cost;       // [Q][gslots]
    double* prob;             // [Q][gslots][D]
    double* fprob;            // [Q][gslots][D]
    double* fprob_sum;        // [Q][D]
    uint32_t* tile_counter;   // [4] work counters of sample_rollouts_dmma_kernel, one per slab of time steps
    unsigned long long* timeline;   // [kTimelineKernels][2] first-CTA-start / last-CTA-end %globaltimer stamps of this iteration, or null
    int32_t rband_halfwidth;  // largest o with R[t][t+o] != 0 (4 for the acceleration rule)
    int32_t r_toeplitz;       // R[t][t+o] does not depend on t (true for R built from the 7-tap rules)
    double r_diag[kRBand + 1]; // r_o = R[t][t+o] when r_toeplitz
    int32_t world_size;
    double* sigma;            // [Q][D]  adapted_stddevs_
    double* coef;             // [Q][D][3] p1, p2, new_stddev of the mean-shifted sampler (PolicyImprovement.cpp:262-269)
    double* updbuf;           // [Q][D][T+2]  update row, numerator and denominator of the noise adaptation (after the all-reduce)
    double* partial;          // [Q][chunks][D][T+2] per-chunk partial sums of weighted_update_kernel
    double* wpart;            // [Q][D][wblocks_cap] per-CTA sums of the unnormalised weights (rollout_weights_kernel)
    double* edge_cost;        // [Q][D][6] control costs of the band-table rows (edge_rows_kernel)
    uint32_t* done_counter;   // [Q][D] tickets of weighted_update_kernel's chunk CTAs (zero between launches)
    double* pt_prob;          // [Q][gslots][D][T] probabilities_ in per-time-step mode (use_cumulative_costs == 0), else null
    double* pt_minden;        // [Q][D][2] min and max(max - min, 1e-8) of the per-time-step costs
    double* s_compact;        // [Q][gslots]    S_k      } compact mirrors of the two columns of `sums` that the weights
    double* c_compact;        // [Q][D][gslots] C_{k,d}  } need, contiguous in k (weights_update_kernel); null when unused
    int32_t wblocks, wblocks_cap;
    int32_t nchunks, chunk;
    double* updates;          // [Q][D][T]    last applied update (read-back)
    double* unit_noise;       // [Q][G][D][T] staging (injected) / debug
    double* epsilon;          // [Q][G][D][T] staging (injected) / debug
    // noise-less rollout record
    double* nl_state;         // [Q][T]
    uint8_t* nl_verdict;      // [Q][T]
    double* nl_control;       // [Q][D][T]
    double* nl_sums;          // [Q][sumw]  record of the noise-less rollout this iteration READS (appended as rollout K)
    double* nl_sums_next;     // [Q][sumw]  record the update of this iteration WRITES for the next one (the two alternate)
    double* nl_total;         // [Q]
    uint8_t* nl_valid;        // [Q]
    double* old_cost;         // [Q]
    double* last_improvement; // [Q]
    double* best_cost;        // [Q]
    int32_t* stop;            // [Q]
    int32_t* iters_used;      // [Q]
    int32_t* note;            // [Q][2] host-mapped pinned progress words (iterations recorded, stopped) written next to iters_used / stop; may be null
    // control-cost operator
    const double* diff_band;  // [rules][N][7]
    const double* Lt;         // [T][T]  Lt[u][t] = L[t][u]
    const double* Rband;      // [T][13] Rband[t][o] = R[t][t-6+o]
    const double* min_stddev; // [D]
    int32_t num_rules;
    int32_t rule_id[kMaxRules];
    double rule_sqrt_w[kMaxRules];
    // one active rule, whose interior rows (3 <= i < N-3) all carry the taps st_dense (offsets -3 .. +3, zeros included):
    // interior_row_cost; otherwise every row walks the band table (band_row_cost) and st_dense is zero
    int32_t st_uniform;
    double st_dense[7];
    // recurrence sampler (sample_rollouts_banded_kernel): rows of L^-1, which is banded — see the kernel's comment
    const double* Lband;      // [T][8]: [0] = 1 / B[t][t], [o] = B[t][t-o] / B[t][t] for o = 1 .. 6 (zero beyond the band / before row 0), [7] unused
    int32_t lband_halfwidth;  // band of B = L^-1 below the diagonal (4 for the acceleration rule); 0 = table not available
    // M-matrix projection (PolicyImprovement::use_projection_, PolicyImprovement.cpp:421-440,706,750-801); all null / 0
    // in the shipped configuration, where M is the identity
    const double* Mproj;      // [T][T] projection_matrix_ = R^-1 with column p scaled by 1 / (T * R^-1[p][p]), row major
    const double* Minv;       // [T][T] inv_projection_matrix_
    double* noise_proj;       // [Q][slots][D][T] noise_projected_ = M * noise_
    const double* rows_noise; // what the control-cost row kernels read: noise (default) or noise_proj
    int32_t rows_mask;        // bit 0: write C_d (control-cost sums), bit 1: write n^T R n; 3 = both (one pass, M = I)
    int32_t per_timestep_minmax;   // per-time-step costs only: min / max per time step (variant at PolicyImprovement.cpp:518-528)
    int32_t noise_from_rollouts;   // the sampler did not write `noise`: weights_update_kernel forms rollouts - theta itself
    // iterations replayed from a CUDA graph (engine.cu: GraphKey) cannot carry per-iteration kernel parameters: the
    // iteration number (Philox counter) and the epoch of the peer exchange then live on the device.  counters[0] =
    // iteration, advanced by the weights / update kernel (nobody reads it any more); counters[1] = exchange epoch, read by
    // weights_update_peer_kernel and advanced by the sampler — reader and writer are never the same launch; counters[2] =
    // the sampler's own iteration number, which every CTA of a launch reads before it takes a ticket in counters[3], the last
    // ticket holder advancing it (so that a sampler that starts under its predecessor never depends on when the
    // predecessor gets to its increment).  Null: the values in `iteration` / PeerExchange::epoch apply.
    uint32_t* counters;
    // forward cumulation (use_cumulative_costs == 2: cumulative_costs_[d](t) = sum_{t' >= t} total_costs_[d](t'), the
    // variant commented out at PolicyImprovement.cpp:473-477): the suffix sums, [Q][slots][D][T]; rides on the
    // per-time-step kernels
    double* pt_cum;
    int32_t forward_cumulation;
    // the recurrence sampler draws and shapes its unit noise (phases 1 and 2) BEFORE it waits for its predecessor: nothing in
    // them depends on what an iteration computes.  Launched as a programmatic dependent of the weights / update kernel, that
    // part runs beside it (sample_rollouts_banded_kernel)
    int32_t early_sampler;
    // [Q] the field of each local query's scene and [Q] its scene (StateKernelArgs::query_sdf), or null: one scene, the
    // kernels' SdfParams argument
    const SdfParams* query_sdf;
    const int32_t* query_scene;
};

// the joint limits of OptimizationTask::filter: all the sampling kernels need of the robot (0.5 KB of kernel parameters
// instead of the 11 KB RobotParams block)
struct JointLimits {
    double lower[STOMP_B200_MAX_DIMS];
    double upper[STOMP_B200_MAX_DIMS];
};

__device__ __forceinline__ bool query_frozen(const LoopParams& p, int q) { return p.honour_stop && p.stop[q] != 0; }

// In-pipeline timeline (stomp_b200_set_timeline): every CTA stamps %globaltimer when it starts and when it ends;
// min / max over the CTAs give the true start and end of each kernel inside the running loop, gaps included —
// which neither ncu (cold caches, serialised) nor event brackets (launch latency) can.
constexpr int kTimelineKernels = 8;   // 0 sample, 1 cost, 2 weights, 3 update, 4 apply, 5 noiseless, 6 reuse, 7 sigma
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// Programmatic dependent launch: the three kernels of a steady iteration (sampler -> state kernel -> weights / update)
// are launched with cudaLaunchAttributeProgrammaticStreamSerialization.  Each lets its successor's CTAs become resident
// at once (trigger at the top) and itself waits for its predecessor's completion and memory flush before it reads
// anything an iteration writes (wait at the top for the state and update kernels: the first thing they read — the stop
// flag — is a predecessor's output; the recurrence sampler first draws and shapes its noise, which depends on nothing an
// iteration computes, and waits before its phase 3).  What is hidden is the launch latency between dependent kernels, 2 - 3 us
// each on B200, and — for the sampler — the part of it that runs beside the update kernel.  Both instructions are no-ops in
// a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_trigger_and_wait()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

struct TimelineScope {
    unsigned long long* slot;
    __device__ __forceinline__ TimelineScope(const LoopParams& p, int kernel) : TimelineScope(p.timeline ? p.timeline + 2 * kernel : nullptr) {}
    __device__ __forceinline__ explicit TimelineScope(unsigned long long* s) : slot(s)
    {
        if (slot && threadIdx.x == 0 && threadIdx.y == 0) atomicMin(slot, global_timer_ns());
    }
    __device__ __forceinline__ void end()
    {
        if (slot) {
            __syncthreads();
            if (threadIdx.x == 0 && threadIdx.y == 0) atomicMax(slot + 1, global_timer_ns());
        }
    }
};

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// block-wide reductions for blockDim.x <= 1024 (scratch: 32 doubles of shared memory); result on all threads
template <int OP>   // 0 sum, 1 min, 2 max
__device__ __forceinline__ double block_reduce(double v, double* scratch)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    v = (OP == 0) ? warp_sum(v) : (OP == 1) ? warp_min(v) : warp_max(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    double r = scratch[0];
    for (int w = 1; w < nwarps; ++w) r = (OP == 0) ? (r + scratch[w]) : (OP == 1) ? fmin(r, scratch[w]) : fmax(r, scratch[w]);
    return r;
}

// parameters of the mean-shifted sampling for one joint (PolicyImprovement.cpp:260-269)
__device__ __forceinline__ void store_sampler_coefficients(const LoopParams& p, int q, int d, double sd)
{
    const double l1 = p.control_cost_weight;
    const double l2 = 1.0 / (sd * sd);
    double* cf = p.coef + ((size_t)q * p.D + d) * 3;
    cf[0] = l1 / (l1 + l2);
    cf[1] = l2 / (l1 + l2);
    cf[2] = 1.0 / sqrt(l1 + l2);
}

// =====================================================================================================
// Philox4x32-10 + Box-Muller
// =====================================================================================================
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key)
{
#pragma unroll
    for (int round = 0; round < 10; ++round) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return ctr;
}

// four standard normals for column `column` (global (query, rollout, joint) index), time steps 4*u4..4*u4+3
__device__ __forceinline__ void philox_normals_keyed(uint2 key, uint32_t iteration, uint32_t column, uint32_t u4, double z[4]);
__device__ __forceinline__ void philox_normals(uint64_t seed, uint32_t iteration, uint32_t column, uint32_t u4, double z[4])
{
    philox_normals_keyed(make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), iteration, column, u4, z);
}
__device__ __forceinline__ void philox_normals_keyed(uint2 key, uint32_t iteration, uint32_t column, uint32_t u4, double z[4])
{
    const uint4 r = philox4x32_10(make_uint4(column, u4, iteration, 0x53544F4Du), key);
    const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u3 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u4f = ((float)(r.w >> 8) + 0.5f) * (1.0f / 16777216.0f);
    // Box-Muller on the SFU (MUFU.LG2 / SIN / COS / RSQ): the library logf / sincospif made this function ~200
    // instructions and 38 % of the sampler's instruction stream (profiles/r1y); the uniforms carry 24 bits, the
    // intrinsics' ~2^-21 absolute error is below that resolution
    // r = sqrt(-2 ln u) = sqrt(-2 ln 2 * log2 u): MUFU.LG2, one multiply, MUFU.SQRT (approximate: no denormal slow path)
    float ra, rb;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(ra) : "f"(-1.3862943611198906f * __log2f(u1)));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rb) : "f"(-1.3862943611198906f * __log2f(u3)));
    float sa, ca, sb, cb;
    __sincosf(6.28318530717958647692f * u2 - 3.14159265358979323846f, &sa, &ca);     // argument in [-pi, pi): the SFU's accurate range
    __sincosf(6.28318530717958647692f * u4f - 3.14159265358979323846f, &sb, &cb);
    z[0] = (double)(ra * ca);
    z[1] = (double)(ra * sa);
    z[2] = (double)(rb * cb);
    z[3] = (double)(rb * sb);
}

// =====================================================================================================
// K1 + K2 + K3: PolicyImprovement::generateRollouts sampling loop (stomp/src/PolicyImprovement.cpp:258-286),
// MultivariateGaussian::sample (stomp/include/stomp/MultivariateGaussian.hpp:91-97), OptimizationTask::filter
// (src/wrappers/stomp/OptimizationTask.cpp:85-106) and computeNoise (PolicyImprovement.cpp:803-810).
// =====================================================================================================

// mean-shifted sample + joint-limit clamp + noise for one element; unit = (L*eps)[t]
__device__ __forceinline__ void shift_clamp_store(const LoopParams& p, const JointLimits& robot, int q, int k, int d, int t,
                                                  double unit)
{
    const double* cf = p.coef + ((size_t)q * p.D + d) * 3;
    const double p1 = cf[0], p2 = cf[1], new_stddev = cf[2];
    const double theta = p.theta_all[((size_t)q * p.D + d) * p.N + kPad + t];
    const double mcc = p.mincc[((size_t)q * p.D + d) * p.T + t];
    double v = p1 * mcc + p2 * theta + new_stddev * unit;
    if (v < robot.lower[d]) v = robot.lower[d];
    if (v > robot.upper[d]) v = robot.upper[d];
    const size_t o = (((size_t)q * p.slots + k) * p.D + d) * p.T + t;
    const double nz = v - theta;
    p.rollouts[o] = v;
    p.noise[o] = nz;
    if (p.proj) p.proj[o] = theta + nz;          // computeProjectedNoise with M = I (PolicyImprovement.cpp:430-440)
    // S_k = sum_t state cost is accumulated with atomics by the state kernel: zeroed here, one element per rollout
    if (d == 0 && t == 0) {
        p.sums[((size_t)q * p.gslots + (p.gen_offset + k)) * p.sumw] = 0.0;
        if (p.s_compact) p.s_compact[(size_t)q * p.gslots + (p.gen_offset + k)] = 0.0;
    }
}

// ---------------------------------------------------------------------------------------------------
// Contraction N^T[c][t] = sum_u E^T[c][u] * Lt[u][t] over the G*D columns c = (k, d) of a query, fused with the
// epilogue above, on the FP64 tensor path (mma.sync.m8n8k4.f64 -> DMMA.8x8x4, the only FP64 MMA shape the hardware has:
// ptxas splits m16n8k16 into eight of them).  Measured on B200 (tools/fp64_peak.cu, profiles/r1_fp64_peak_b200.json):
// DMMA 37.0 TFLOP/s vs 35.0 TFLOP/s on the FMA pipe — the same peak, but one DMMA carries the work of eight DFMA
// warp-instructions, and ncu showed the earlier FMA-pipe version of this contraction issue-bound, i.e. the case
// BASELINE.json's north_star reserves tensor cores for.
//
// Per warp: one m8 tile = 8 columns (k, d) x all time steps of a 104-wide slab of t; C = 13 n8 tiles in registers;
// B = the Lt slab, resident in shared memory for the whole kernel; tiles handed out by an atomic counter (reset
// by the state kernel) over the flattened (query, rollout, joint) column space.
// A = eps never touches memory: lane (r, kq) draws the four normals eps[column r][u0 + 4kq .. + 3] with one
// Philox call per 16-wide chunk of u, and the contraction index is PERMUTED inside the chunk so that they are
// exactly its A fragments: in step j of the chunk, k-slot kq stands for u = u0 + 4kq + j, i.e. A = z[j] and
// B = Lt[u0 + 4kq + j][t].  (A sum over u does not care about the order of u.)  The slab's row stride is
// 106 == 2 (mod 4) doubles, which puts the four rows 4kq + j of a B fragment on disjoint banks (2 wavefronts
// per load, the minimum for 64-bit lanes).
// Lt is upper triangular: a chunk only touches n8 tiles with 8 nt + 7 >= u0 - t_base; the first tile is a
// template argument (13 straight-line bodies behind one switch), so the inner loop is LDS + DMMA with no
// predicates.  The epilogue holds two consecutive time steps per lane and n8 tile: 16-byte loads / stores.
// ---------------------------------------------------------------------------------------------------
// kTiles n8 tiles per slab (template argument: 13 for T = 100 / 200, 10 for T = 150, fewer for short trajectories —
// the slabs of a launch are equally wide, so no warp multiplies against zero columns and short trajectories keep
// fewer accumulators and more warps per SM)
constexpr int kDmmaWarps = 8;
constexpr int kSlabTilesMax = 13;
__host__ __device__ constexpr int dmma_slab_stride(int tiles) { return 8 * tiles + 2; }     // == 2 (mod 4)

__host__ __device__ constexpr int dmma_slab_rows(int T) { return (T + 15) & ~15; }

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int kFirstTile, int kTiles>
__device__ __forceinline__ void dmma_chunk(double (&acc)[kTiles][2], const double (&z)[4], const double* __restrict__ b0)
{
    constexpr int kSlabStride = dmma_slab_stride(kTiles);
    if constexpr (kFirstTile < kTiles) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int nt = kFirstTile; nt < kTiles; ++nt) dmma_m8n8k4(acc[nt][0], acc[nt][1], z[j], b0[j * kSlabStride + 8 * nt]);
        }
    }
}

template <int kTiles, bool kPhilox>
__global__ void __launch_bounds__(kDmmaWarps * 32)
sample_rollouts_dmma_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ JointLimits robot,
                            unsigned* __restrict__ tile_counter)
{
    extern __shared__ double smem[];
    constexpr int kSlabTiles = kTiles;
    constexpr int kSlabT = 8 * kTiles;
    constexpr int kSlabStride = dmma_slab_stride(kTiles);
    const int T = p.T, D = p.D, N = p.N;
    const int rows = dmma_slab_rows(T);
    const int slab = blockIdx.y;
    const int t_base = slab * kSlabT;
    const int u_end = min(rows, dmma_slab_rows(min(T, t_base + kSlabT)));   // rows of Lt below the slab's last t are zero
    const int tid = threadIdx.x, lane = tid & 31;
    TimelineScope tls(p, 0);
    double* sLt = smem;                                              // [rows][kSlabStride]; zero outside the matrix

    if ((T & 1) == 0) {
        // 16-byte copies, eight in flight per thread: the fill is pure L2 latency (it was a quarter of the kernel's
        // stall samples as a one-load-per-iteration loop, profiles/r1u)
        constexpr int kPairs = kSlabStride / 2;        // 53 pairs per row, the last one padding
        const int npairs = rows * kPairs;
#pragma unroll 8
        for (int e = tid; e < npairs; e += kDmmaWarps * 32) {
            const int u = e / kPairs, j = 2 * (e - u * kPairs), t = t_base + j;
            double2 v = make_double2(0.0, 0.0);
            if (u < T && j < kSlabT && t < T && t + 1 >= u) {
                v = *reinterpret_cast<const double2*>(p.Lt + (size_t)u * T + t);
                if (t < u) v.x = 0.0;
            }
            *reinterpret_cast<double2*>(sLt + (size_t)u * kSlabStride + j) = v;
        }
    } else {
#pragma unroll 8
        for (int e = tid; e < rows * kSlabStride; e += kDmmaWarps * 32) {
            const int u = e / kSlabStride, j = e - u * kSlabStride, t = t_base + j;
            sLt[e] = (u < T && j < kSlabT && t < T && t >= u) ? p.Lt[(size_t)u * T + t] : 0.0;
        }
    }
    __syncthreads();

    const int ncols = p.num_gen * D;                  // columns per query
    const long long total_cols = (long long)p.Q * ncols;
    const int ntiles = (int)((total_cols + 7) >> 3);
    const int r = lane >> 2, kq = lane & 3;
    const bool pairs = (T & 1) == 0;                  // 16-byte epilogue: every row starts on an even element
    for (;;) {
        int tile = 0;
        if (lane == 0) tile = (int)atomicAdd(tile_counter + slab, 1u);
        tile = __shfl_sync(0xffffffffu, tile, 0);
        if (tile >= ntiles) break;
        const long long cg = (long long)tile * 8 + r;  // this lane's column (row of the m8 tile)
        const bool in_range = cg < total_cols;
        const int q = in_range ? (int)(cg / ncols) : 0;
        const int c = in_range ? (int)(cg - (long long)q * ncols) : 0;
        const int k = c / D, d = c - k * D;
        const bool live = in_range && !query_frozen(p, q);
        const size_t gen_row = (((size_t)q * p.num_gen + k) * D + d) * T;     // row of the [Q][G][D][T] staging tensors
        const uint32_t gcol = (uint32_t)((((size_t)(p.query_offset + q)) * p.gen_global + (p.gen_offset + k)) * D + d);

        double acc[kSlabTiles][2];
#pragma unroll
        for (int nt = 0; nt < kSlabTiles; ++nt) { acc[nt][0] = 0.0; acc[nt][1] = 0.0; }

        for (int u0 = 0; u0 < u_end; u0 += 16) {
            // ---- eps[column][u0 + 4kq .. + 3]: the A fragments of the chunk's four steps ----
            double z[4] = {0.0, 0.0, 0.0, 0.0};
            const int ub = u0 + 4 * kq;
            if (live) {
                if (kPhilox) {
                    philox_normals(p.seed, (uint32_t)p.iteration, gcol, (uint32_t)(ub >> 2), z);
                    if (p.store_unit && slab == (int)gridDim.y - 1) {      // the last slab walks every u < T
#pragma unroll
                        for (int m = 0; m < 4; ++m)
                            if (ub + m < T) p.epsilon[gen_row + ub + m] = z[m];
                    }
                } else {
#pragma unroll
                    for (int m = 0; m < 4; ++m)
                        if (ub + m < T) z[m] = p.epsilon[gen_row + ub + m];
                }
#pragma unroll
                for (int m = 0; m < 4; ++m)
                    if (ub + m >= T) z[m] = 0.0;
            }
            const double* b0 = sLt + (size_t)ub * kSlabStride + r;
            switch (u0 > t_base ? (u0 - t_base) >> 3 : 0) {      // warp-uniform
                case 0: dmma_chunk<0, kTiles>(acc, z, b0); break;
                case 1: dmma_chunk<1, kTiles>(acc, z, b0); break;
                case 2: dmma_chunk<2, kTiles>(acc, z, b0); break;
                case 3: dmma_chunk<3, kTiles>(acc, z, b0); break;
                case 4: dmma_chunk<4, kTiles>(acc, z, b0); break;
                case 5: dmma_chunk<5, kTiles>(acc, z, b0); break;
                case 6: dmma_chunk<6, kTiles>(acc, z, b0); break;
                case 7: dmma_chunk<7, kTiles>(acc, z, b0); break;
                case 8: dmma_chunk<8, kTiles>(acc, z, b0); break;
                case 9: dmma_chunk<9, kTiles>(acc, z, b0); break;
                case 10: dmma_chunk<10, kTiles>(acc, z, b0); break;
                case 11: dmma_chunk<11, kTiles>(acc, z, b0); break;
                default: dmma_chunk<12, kTiles>(acc, z, b0); break;
            }
        }
        // ---- epilogue: C fragment element (row r, cols 2*kq, 2*kq + 1) of tile nt ----
        if (!live) continue;
        if (pairs) {
            const double* cf = p.coef + ((size_t)q * D + d) * 3;
            const double p1 = cf[0], p2 = cf[1], new_stddev = cf[2];
            const double lo = robot.lower[d], hi = robot.upper[d];
            const double* th = p.theta_all + ((size_t)q * D + d) * N + kPad;
            const double* mc = p.mincc + ((size_t)q * D + d) * T;
            const size_t row = (((size_t)q * p.slots + k) * D + d) * T;
            // batches of four n8 tiles: the eight 16-byte loads of a batch are issued together (left to the compiler they
            // were issued one tile at a time, each exposing an L1 / L2 round trip to the four resident warps)
#pragma unroll
            for (int nb = 0; nb < kSlabTiles; nb += 4) {
                double2 th2[4], mc2[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int t = t_base + 8 * (nb + i) + 2 * kq;
                    th2[i] = make_double2(0.0, 0.0); mc2[i] = make_double2(0.0, 0.0);
                    if (nb + i < kSlabTiles && t < T) {
                        th2[i] = *reinterpret_cast<const double2*>(th + t);
                        mc2[i] = *reinterpret_cast<const double2*>(mc + t);
                    }
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int nt = nb + i;
                    const int t = t_base + 8 * nt + 2 * kq;
                    if (nt < kSlabTiles && t < T) {
                        // the arithmetic of shift_clamp_store, two time steps at once
                        double v0 = p1 * mc2[i].x + p2 * th2[i].x + new_stddev * acc[nt < kSlabTiles ? nt : 0][0];
                        double v1 = p1 * mc2[i].y + p2 * th2[i].y + new_stddev * acc[nt < kSlabTiles ? nt : 0][1];
                        if (v0 < lo) v0 = lo;
                        if (v0 > hi) v0 = hi;
                        if (v1 < lo) v1 = lo;
                        if (v1 > hi) v1 = hi;
                        const double n0 = v0 - th2[i].x, n1 = v1 - th2[i].y;
                        *reinterpret_cast<double2*>(p.rollouts + row + t) = make_double2(v0, v1);
                        *reinterpret_cast<double2*>(p.noise + row + t) = make_double2(n0, n1);
                        if (p.proj) *reinterpret_cast<double2*>(p.proj + row + t) = make_double2(th2[i].x + n0, th2[i].y + n1);
                        if (p.store_unit)
                            *reinterpret_cast<double2*>(p.unit_noise + gen_row + t) =
                                make_double2(acc[nt < kSlabTiles ? nt : 0][0], acc[nt < kSlabTiles ? nt : 0][1]);
                        if (d == 0 && t == 0) {
                            p.sums[((size_t)q * p.gslots + (p.gen_offset + k)) * p.sumw] = 0.0;
                            if (p.s_compact) p.s_compact[(size_t)q * p.gslots + (p.gen_offset + k)] = 0.0;
                        }
                    }
                }
            }
        } else {
#pragma unroll
            for (int nt = 0; nt < kSlabTiles; ++nt) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int t = t_base + 8 * nt + 2 * kq + h;
                    if (t < T) {
                        if (p.store_unit) p.unit_noise[gen_row + t] = acc[nt][h];
                        shift_clamp_store(p, robot, q, k, d, t, acc[nt][h]);
                    }
                }
            }
        }
    }
    tls.end();
}

// ---------------------------------------------------------------------------------------------------
// PolicyImprovement::computeProjectedNoise (PolicyImprovement.cpp:421-440) with use_projection_:
//   noise_projected_[c][t] = sum_u M[t][u] * noise_[c][u],  parameters_noise_projected_ = parameters_ + noise_projected_
// for the G * D generated columns c = (k, d) of every query: the second contraction of the loop, dense this time (M =
// R^-1 with scaled columns), on the same FP64 tensor path as the sampler (mma.sync.m8n8k4.f64).  CTA tile 32 columns x
// 64 time steps, four warps of 8 columns each (8 n8 tiles = 16 accumulators), u walked in chunks of 16 through two
// shared-memory tiles; reads `noise` (after the joint-limit clamp: the clamp is why this is not folded into L).
// Not a shipped configuration (the reference constructs use_projection_ = false, PolicyImprovement.cpp:57): built for
// completeness and correctness, sized so that it never dominates (2 x the sampler's flops).
// grid (ceil(G D / 32), ceil(T / 64), Q), 128 threads.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
project_noise_dmma_kernel(const __grid_constant__ LoopParams p)
{
    constexpr int BM = 32, BN = 64, BK = 16;
    __shared__ double As[BM][BK + 2];        // As[c][u]; the + 2 keeps the four k-slots of a fragment on different banks
    __shared__ double Bs[BK][BN + 2];        // Bs[u][t] = M[t0 + t][u0 + u]
    const int q = blockIdx.z;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D;
    const int ncols = p.num_gen * D;
    const int c0 = blockIdx.x * BM, t0 = blockIdx.y * BN;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = lane >> 2, kq = lane & 3;
    const double* nz = p.noise + (size_t)q * p.slots * D * T;      // rows c of [slots * D][T]; generated rows come first
    double acc[8][2];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) { acc[nt][0] = 0.0; acc[nt][1] = 0.0; }
    for (int u0 = 0; u0 < T; u0 += BK) {
        for (int e = tid; e < BM * BK; e += 128) {
            const int c = e / BK, u = e - c * BK;
            As[c][u] = (c0 + c < ncols && u0 + u < T) ? nz[(size_t)(c0 + c) * T + u0 + u] : 0.0;
        }
        for (int e = tid; e < BK * BN; e += 128) {
            const int t = e / BK, u = e - t * BK;           // consecutive threads walk u: M rows are contiguous in u
            Bs[u][t] = (t0 + t < T && u0 + u < T) ? p.Mproj[(size_t)(t0 + t) * T + u0 + u] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < BK / 4; ++j) {
            const double a = As[warp * 8 + r][4 * j + kq];
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) dmma_m8n8k4(acc[nt][0], acc[nt][1], a, Bs[4 * j + kq][8 * nt + r]);
        }
        __syncthreads();
    }
    const int c = c0 + warp * 8 + r;
    if (c < ncols) {
        const int k = c / D, d = c - k * D;
        const size_t row = (((size_t)q * p.slots + k) * D + d) * T;
        const double* th = p.theta_all + ((size_t)q * D + d) * p.N + kPad;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int t = t0 + 8 * nt + 2 * kq + h;
                if (t < T) {
                    p.noise_proj[row + t] = acc[nt][h];
                    if (p.proj) p.proj[row + t] = th[t] + acc[nt][h];
                }
            }
    }
}

// ---- control costs: CovariantMovementPrimitive::computeControlCosts (stomp/src/CovariantMovementPrimitive.cpp:
// 363-377): costs_all[i] = sum_rules dt*w*(Ax*Ax), Ax = (D_rule x)[i] * sqrt(w_rule).  Every kernel that forms a row, an
// n^T R n term or a write-back of the sums does it through the functions of this section.
// Band-table row i: every active rule, columns max(0, i-3) .. min(N-1, i+3) in order.  x(j) = x_all[j] (a shared-memory or a
// global row).
template <class X>
__device__ __forceinline__ double band_row_cost(const LoopParams& p, int i, X x)
{
    const double dtw = p.dt * p.control_cost_weight;
    double c = 0.0;
    for (int r = 0; r < p.num_rules; ++r) {
        const double* band = p.diff_band + ((size_t)p.rule_id[r] * p.N + i) * 7;
        double s = 0.0;
        const int lo = max(0, i - 3), hi = min(p.N - 1, i + 3);
        for (int j = lo; j <= hi; ++j) s += __ldg(band + (j - i + 3)) * x(j);
        const double Ax = s * p.rule_sqrt_w[r];
        c += dtw * (Ax * Ax);
    }
    return c;
}

// Interior row (3 <= i < N-3) of the single active rule (p.st_uniform): the taps st_dense[kLo .. kHi], the others being
// zero, multiplied then added in column order — the reference's arithmetic; a zero tap adds an exact zero, so any kLo / kHi
// that covers the non-zero taps gives the same bits.  x(o) = x_all[i - 3 + o].
template <int kLo, int kHi, class X>
__device__ __forceinline__ double interior_row_cost(const LoopParams& p, X x)
{
    double s = 0.0;
#pragma unroll
    for (int o = kLo; o <= kHi; ++o) s += p.st_dense[o] * x(o);
    const double Ax = s * p.rule_sqrt_w[0];
    return (p.dt * p.control_cost_weight) * (Ax * Ax);
}

// either of the two above, for row i of a row held in memory (x[j] = x_all[j])
__device__ __forceinline__ double control_cost_row(const LoopParams& p, const double* x, int i)
{
    if (p.st_uniform && i >= 3 && i < p.N - 3) return interior_row_cost<0, 6>(p, [&](int o) { return x[i - 3 + o]; });
    return band_row_cost(p, i, [&](int j) { return x[j]; });
}

// The n^T R n term of time step t (PolicyImprovement.cpp:656-663): n_t (R_tt n_t + 2 sum_{o=1..kB} R_{t,t+o} n_{t+o}); R is
// symmetric and banded, so each pair counts once.  r[o] = R_{t,t+o}: the Toeplitz diagonals r_diag or the row of Rband at t;
// n(o) = noise[t + o], zero outside [0, T).
template <int kB, class Nz>
__device__ __forceinline__ double quad_term(const double* r, Nz n)
{
    double s = 0.0;
#pragma unroll
    for (int o = 1; o <= kB; ++o) s += r[o] * n(o);
    return n(0) * (r[0] * n(0) + 2.0 * s);
}

// the six padding-only rows of (query, joint), summed (edge_rows_kernel leaves them in edge_cost)
__device__ __forceinline__ double edge_cost_sum(const LoopParams& p, int q, int d)
{
    const double* ec = p.edge_cost + ((size_t)q * p.D + d) * 6;
    return ((ec[0] + ec[1]) + (ec[2] + ec[3])) + (ec[4] + ec[5]);
}

// C_d and n^T R n of generated rollout k into `sums` (and C_d into c_compact), as far as rows_mask asks
__device__ __forceinline__ void store_row_sums(const LoopParams& p, int q, int k, int d, double C_d, double quad)
{
    double* srow = p.sums + ((size_t)q * p.gslots + (p.gen_offset + k)) * p.sumw;
    if (p.rows_mask & 1) {
        srow[1 + d] = C_d;
        if (p.c_compact) p.c_compact[((size_t)q * p.D + d) * p.gslots + (p.gen_offset + k)] = C_d;
    }
    if (p.rows_mask & 2) srow[1 + 2 * p.D + d] = p.use_noise_adaptation ? quad : 0.0;
}

// One (rollout, joint) row for one warp: C_d = sum of the per-timestep control costs (padding rows folded into
// the first / last free step, i.e. simply included in the sum) and cum_d = sum_t (state + control).
// x: padded trajectory of this (rollout, joint) in shared memory; state: state costs [T] in shared memory.
__device__ __forceinline__ void control_cost_sums(const LoopParams& p, const double* x, const double* state, int lane,
                                                  double& C_d, double& cum_d)
{
    const int T = p.T, N = p.N;
    double c_sum = 0.0, s_sum = 0.0;
    for (int i = lane; i < N; i += 32) {
        c_sum += control_cost_row(p, x, i);
        if (state && i < T) s_sum += state[i];
    }
    c_sum = warp_sum(c_sum);
    s_sum = warp_sum(s_sum);
    C_d = c_sum;
    cum_d = s_sum + c_sum;
}

// per-timestep control costs in the reference's layout and folding order (:363-377); read-backs / noise-less record
__device__ __forceinline__ void control_cost_store(const LoopParams& p, const double* x, int lane, double* control_out /*[T]*/)
{
    const int T = p.T, N = p.N;
    for (int t = lane; t < T; t += 32) control_out[t] = control_cost_row(p, x, kPad + t);
    // the 2 * kPad padding rows: one lane each (twelve dependent table walks on one lane were most of the noise-less
    // kernel's time), then lane 0 adds them in the reference's order
    double v = 0.0;
    if (lane < 2 * kPad) v = control_cost_row(p, x, lane < kPad ? lane : N - (lane - kPad + 1));
    __syncwarp();
    double first = (lane == 0) ? control_out[0] : 0.0, last = (lane == 0) ? control_out[T - 1] : 0.0;
#pragma unroll
    for (int i = 0; i < kPad; ++i) {
        first += __shfl_sync(0xffffffffu, v, i);
        last += __shfl_sync(0xffffffffu, v, kPad + i);
    }
    if (lane == 0) {
        control_out[0] = first;
        control_out[T - 1] = last;
    }
}

// ---------------------------------------------------------------------------------------------------
// The same sample without the contraction.  L = chol(R^-1) (MultivariateGaussian.hpp:81) is dense, but its INVERSE is
// banded: factor the banded R = U U^T with U UPPER triangular (a Cholesky factorisation run from the last row up; U has R's
// half bandwidth b, 4 for the shipped acceleration rule).  Then R^-1 = U^-T U^-1 with U^-T lower triangular and positive
// on the diagonal, and the Cholesky factor is unique, so L = U^-T exactly and
//     n = L eps   <=>   U^T n = eps   <=>   n_t = (eps_t - sum_{o=1..b} U[t-o][t] n_{t-o}) / U[t][t]:
// a b-term recurrence per column, O(T b) instead of the O(T^2 / 2) contraction — 65 x fewer FP64 operations at T = 100,
// and the FP64 pipe is what bounds this loop (DMMA and DFMA share it: tools/fp64_mixed.cu, profiles/r3_fp64_mixed.json).
// It is also the more accurate statement of the same map: against a long-double solve the recurrence is good to 1e-14,
// while L as the reference computes it (fullPivLu().inverse() then llt(), cond(R) = 6e6 at T = 100) carries 7e-11 — the
// two agree to that 7e-11 (3e-10 at T = 200), inside the 1e-9 bar; tests/test_gpu_parity.py holds both statements.
// The host builds the table from R (engine.cu: build_sampler_band) and checks it against the L it was given; injected
// epsilon (parity mode) and matrices that fail the check go through the DMMA contraction above with the caller's L.
//
// Mapping: one CTA (four warps) = 32 rollouts of ONE joint of one query; the 32 x T tile of eps / unit noise / samples
// lives in shared memory (odd row stride: walks along t by one lane per rollout and walks along t by consecutive lanes
// are both conflict free).  Phases, separated by CTA barriers; seven CTAs per SM keep 28 warps in flight:
//   1. eps: lane = rollout, the warps share the groups of four time steps — same Philox counters as the contraction
//      kernels, so the same seed gives the same eps — or copy the injected eps;
//   2. the recurrence: warp 0, lane = rollout, sequential in t, band rows of L^-1 from a shared-memory table; the n_{t-1}
//      term is the only one on the critical path;
//   3a. lane = rollout again, each warp a quarter of the time steps, sequential in t: mean shift p1 * mincc + p2 * theta +
//      new_stddev * n, joint-limit clamp (the sample replaces the unit noise in the tile), noise = clamped - theta, and —
//      kFuse — the control-cost stencil and n^T R n from a 5-wide window of the noise that slides through REGISTERS (the
//      six noise values a quarter needs from its neighbours are taken before anyone overwrites the tile): K5 / K6 cost
//      no pass over `noise` in HBM, no kernel of their own, no shuffle.  The stencil uses linearity:
//      (D x)_i = (D theta_all)_i + sum_m c_m noise[i - 8 + m], the first term a per-CTA table;
//   3b. lane = time step: the tile leaves as coalesced rows of `rollouts` and `noise` (= sample - theta).
// kFuse needs the shipped shape of the operator (one 5-tap rule, Toeplitz R with half bandwidth <= 4); otherwise the row
// kernels run afterwards.  kB: band of the recurrence, 4 or 6.
// ---------------------------------------------------------------------------------------------------
constexpr int kBandedThreads = 128;
__host__ __device__ inline int banded_tile_stride(int T) { return T | 1; }
__host__ __device__ inline int banded_band_doubles(int T, int kB) { return (T * (kB + 1) > 256 + 2 * T) ? T * (kB + 1) : 256 + 2 * T; }
__host__ __device__ inline size_t banded_sampler_smem_doubles(int T, int N, int kB)
{
    // tile [32][T | 1] | band [T][kB + 1], reused after phase 2 for [256] partial sums + mean [T] + theta [T] | (D theta_all)_i [N].
    // 30.8 KB at T = 100: SEVEN CTAs per SM, which is what the 896 tiles of BASELINE config 3 need to be one wave on 148 SMs
    return (size_t)32 * banded_tile_stride(T) + (size_t)banded_band_doubles(T, kB) + (size_t)N;
}

template <int kB, bool kPhilox, bool kFuse>
__global__ void __launch_bounds__(kBandedThreads, 7)
sample_rollouts_banded_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ JointLimits robot)
{
    extern __shared__ __align__(16) double smem[];
    const int q = blockIdx.y;
    // Phases 1 and 2 (Philox + Box-Muller, the recurrence: two thirds of this kernel's instructions) read nothing an iteration
    // writes — band table, seed, iteration number — so with `early` the wait for the predecessor (the weights / update
    // kernel of the previous iteration, when this launch is its programmatic dependent) comes after them: the CTAs become
    // resident at the predecessor's trigger and work beside a kernel that leaves four fifths of the warp slots empty.
    const bool early = kPhilox && p.early_sampler != 0;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    uint32_t iteration = (uint32_t)p.iteration;
    if (p.counters) {
        iteration = *(volatile const uint32_t*)(p.counters + 2);
        __syncthreads();                                     // every thread of the CTA has its copy
        if (threadIdx.x == 0) {
            __threadfence();
            const unsigned ticket = atomicAdd(p.counters + 3, 1u);
            if (ticket == gridDim.x * gridDim.y - 1u) {      // every CTA of this launch has read counters[2]
                p.counters[3] = 0u;
                p.counters[2] = iteration + 1u;
            }
        }
    }
    if (!early) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (p.counters && blockIdx.x == 0 && q == 0 && threadIdx.x == 0) p.counters[1] += 1u;    // next exchange epoch (graph replay)
        if (query_frozen(p, q)) return;
    }
    TimelineScope tls(p, 0);
    const int T = p.T, D = p.D, N = p.N;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nkb = (p.num_gen + 31) >> 5;
    const int d = blockIdx.x / nkb, kb = blockIdx.x - d * nkb;
    const int k0 = kb * 32;
    const int ncol = min(32, p.num_gen - k0);                // live rollouts of this tile
    const int S = banded_tile_stride(T);
    const bool debug_stores = p.store_unit != 0;
    const bool live = lane < ncol;                           // lane = rollout phases

    double* s_tile = smem;                                   // [32][S]
    double* s_band = s_tile + 32 * S;                        // [T][kB + 1]: 1 / B_tt, B_{t,t-1} / B_tt, ...
    double* s_dth = s_band + banded_band_doubles(T, kB);     // [N]  (D theta_all)_i for the interior rows 3 .. N-4
    double* s_part = s_band;                                 // after phase 2 the band table is dead: [2][4][32] partial sums of phase 3a,
    double* s_mean = s_band + 256;                           //   [T] p1 * mincc + p2 * theta (the first two terms of the mean-shifted sample)
    double* s_th = s_mean + T;                               //   [T] theta
    const double* th_all = p.theta_all + ((size_t)q * D + d) * N;
    const double* mc_row = p.mincc + ((size_t)q * D + d) * T;
    const double c1 = p.st_dense[1], c2 = p.st_dense[2], c3 = p.st_dense[3], c4 = p.st_dense[4], c5 = p.st_dense[5];
    for (int i = tid; i < T * (kB + 1); i += kBandedThreads) {
        const int t = i / (kB + 1), o = i - t * (kB + 1);
        s_band[i] = p.Lband[t * 8 + o];
    }
    // ---- phase 1: eps ----
    if (live) {
        const int ngroups = (T + 3) >> 2;
        // global column of this rollout and joint: the Philox counter of the contraction kernels
        const uint32_t gcol = (uint32_t)(((uint32_t)(p.query_offset + q) * (uint32_t)p.gen_global + (uint32_t)(p.gen_offset + k0 + lane)) * (uint32_t)D + (uint32_t)d);
        const uint2 key = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
        double* dst = s_tile + lane * S;
        double* eps_row = p.epsilon + (((size_t)q * p.num_gen + (k0 + lane)) * D + d) * T;
        for (int g = warp; g < ngroups; g += kBandedThreads / 32) {
            const int tg = 4 * g;
            double z[4];
            if (kPhilox) {
                philox_normals_keyed(key, iteration, gcol, (uint32_t)g, z);
                if (debug_stores) {
#pragma unroll
                    for (int m = 0; m < 4; ++m)
                        if (tg + m < T) eps_row[tg + m] = z[m];
                }
            } else {
#pragma unroll
                for (int m = 0; m < 4; ++m) z[m] = (tg + m < T) ? eps_row[tg + m] : 0.0;
            }
            if (tg + 3 < T) { dst[tg] = z[0]; dst[tg + 1] = z[1]; dst[tg + 2] = z[2]; dst[tg + 3] = z[3]; }
            else {
#pragma unroll
                for (int m = 0; m < 4; ++m)
                    if (tg + m < T) dst[tg + m] = z[m];
            }
        }
    }
    __syncthreads();
    // ---- phase 2: the recurrence, in place (eps -> unit noise) ----
    if (warp == 0 && live) {
        double h[kB];
#pragma unroll
        for (int o = 0; o < kB; ++o) h[o] = 0.0;
        double* col = s_tile + lane * S;
        // Blocks of four steps: every shared-memory load of the block (eps of this rollout, warp-uniform band rows) is issued
        // before its first store — the compiler cannot prove that `col` and the band table do not alias and would otherwise
        // expose a shared-memory round trip per step (measured: 88 cycles per step, 4.5 us per tile).  Inside a block the
        // terms of n_{t-2} .. n_{t-kB} come first and n_{t-1} last: one DFMA per step on the critical path.
        int t = 0;
        for (; t + 4 <= T; t += 4) {
            double e[4], bb[4][kB + 1];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                e[m] = col[t + m];
#pragma unroll
                for (int o = 0; o <= kB; ++o) bb[m][o] = s_band[(t + m) * (kB + 1) + o];
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                double acc = e[m] * bb[m][0];
#pragma unroll
                for (int o = kB - 1; o >= 0; --o) acc = fma(-bb[m][1 + o], h[o], acc);
#pragma unroll
                for (int o = kB - 1; o > 0; --o) h[o] = h[o - 1];
                h[0] = acc;
                e[m] = acc;
            }
#pragma unroll
            for (int m = 0; m < 4; ++m) col[t + m] = e[m];
        }
        for (; t < T; ++t) {
            const double* b = s_band + t * (kB + 1);
            double acc = col[t] * b[0];
#pragma unroll
            for (int o = kB - 1; o >= 0; --o) acc = fma(-b[1 + o], h[o], acc);
#pragma unroll
            for (int o = kB - 1; o > 0; --o) h[o] = h[o - 1];
            h[0] = acc;
            col[t] = acc;
        }
    }
    if (early) {                                             // from here on: the parameters and scales the previous iteration left
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (p.counters && blockIdx.x == 0 && q == 0 && threadIdx.x == 0) p.counters[1] += 1u;    // next exchange epoch (graph replay)
        if (query_frozen(p, q)) return;
    }
    __syncthreads();
    // ---- phase 3a: lane = rollout, warp w = time steps [a, b) ----
    const double* cf = p.coef + ((size_t)q * D + d) * 3;
    const double p1 = cf[0], p2 = cf[1], sd = cf[2];
    if (kFuse)
        for (int i = tid; i < N; i += kBandedThreads) {
            double v = 0.0;
            if (i >= 3 && i < N - 3) {
                v = c1 * th_all[i - 2];
                v = fma(c2, th_all[i - 1], v); v = fma(c3, th_all[i], v); v = fma(c4, th_all[i + 1], v); v = fma(c5, th_all[i + 2], v);
            }
            s_dth[i] = v;
        }
    for (int t = tid; t < T; t += kBandedThreads) {
        const double th = th_all[kPad + t];
        s_th[t] = th;
        s_mean[t] = p1 * mc_row[t] + p2 * th;
    }
    __syncthreads();
    const double lo = robot.lower[d], hi = robot.upper[d];
    const double r0 = p.r_diag[0], r1 = 2.0 * p.r_diag[1], r2 = 2.0 * p.r_diag[2], r3 = 2.0 * p.r_diag[3], r4 = 2.0 * p.r_diag[4];
    const int Tq = (T + 3) >> 2;
    const int a = warp * Tq, b = min(T, a + Tq);
    const bool has_steps = a < T;
    const bool last = has_steps && b == T;
    double* col = s_tile + lane * S;
    // clamped sample for unit noise `unit` at time step s: the arithmetic of shift_clamp_store (PolicyImprovement.cpp:262-269)
    auto sample_of = [&](int s, double unit, double& theta) {
        theta = s_th[s];
        double v = s_mean[s] + sd * unit;
        if (v < lo) v = lo;
        if (v > hi) v = hi;
        return v;
    };
    // noise values this quarter needs from its neighbours (4 behind, 2 ahead), taken before the tile is overwritten
    double hm4 = 0.0, hm3 = 0.0, hm2 = 0.0, hm1 = 0.0, hp0 = 0.0, hp1 = 0.0;
    if (kFuse && has_steps && live) {
        double th;
        if (a - 4 >= 0) hm4 = sample_of(a - 4, col[a - 4], th) - th;
        if (a - 3 >= 0) hm3 = sample_of(a - 3, col[a - 3], th) - th;
        if (a - 2 >= 0) hm2 = sample_of(a - 2, col[a - 2], th) - th;
        if (a - 1 >= 0) hm1 = sample_of(a - 1, col[a - 1], th) - th;
        if (b < T) hp0 = sample_of(b, col[b], th) - th;
        if (b + 1 < T) hp1 = sample_of(b + 1, col[b + 1], th) - th;
    }
    if (debug_stores) {                                      // read-backs of the unit noise (parity tests): rows of the tile as they are now
        for (int c = warp * 8; c < min(warp * 8 + 8, ncol); ++c) {
            double* unit_row = p.unit_noise + (((size_t)q * p.num_gen + (k0 + c)) * D + d) * T;
            for (int t = lane; t < T; t += 32) unit_row[t] = s_tile[c * S + t];
        }
    }
    __syncthreads();
    double ss = 0.0, quad = 0.0;
    if (has_steps && live) {
        double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0, w4 = 0.0;     // noise[s-4 .. s]
        // noise[s] enters the window: row i = (s - 2) + 6 of the differentiation matrix is complete, and so is the n^T R n term of s
        auto push = [&](double nz, int s, bool row, bool term) {
            w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = nz;
            if (row) {
                double sacc = s_dth[s - 2 + kPad];
                sacc = fma(c1, w0, sacc); sacc = fma(c2, w1, sacc); sacc = fma(c3, w2, sacc); sacc = fma(c4, w3, sacc); sacc = fma(c5, w4, sacc);
                ss = fma(sacc, sacc, ss);
            }
            if (term) {
                double qs = r0 * w4;
                qs = fma(r1, w3, qs); qs = fma(r2, w2, qs); qs = fma(r3, w1, qs); qs = fma(r4, w0, qs);
                quad = fma(w4, qs, quad);                    // n_s (R_ss n_s + 2 sum_{o>0} R_{s,s-o} n_{s-o}): each pair once; zero outside [0, T)
            }
        };
        // rows t' = s - 2 owned by this quarter: [a, b); the first quarter also -3 .. -1 (start padding), the last one also
        // T .. T + 2 (goal padding)
        const int own_lo = (a == 0) ? -3 : a, own_hi = last ? T + 3 : b;
        auto owns = [&](int s) { return s - 2 >= own_lo && s - 2 < own_hi; };
        if (kFuse) {
            push(hm4, a - 4, false, false); push(hm3, a - 3, false, false); push(hm2, a - 2, false, false);
            push(hm1, a - 1, owns(a - 1), false);            // s = -1 completes row -3 (all-zero noise)
        }
        int s = a;
        // the first two steps complete rows of the previous quarter (unless this is the first one): generic path
        for (; s < min(a + 2, b); ++s) {
            double theta;
            const double v = sample_of(s, col[s], theta);
            col[s] = v;
            if (kFuse) push(v - theta, s, owns(s), true);
        }
        // blocks of five steps (the window's rotation period: no register moves), loads before stores as in phase 2
        for (; s + 5 <= b; s += 5) {
            double u[5], th[5], mn[5], dt5[5];
#pragma unroll
            for (int m = 0; m < 5; ++m) { u[m] = col[s + m]; th[m] = s_th[s + m]; mn[m] = s_mean[s + m]; if (kFuse) dt5[m] = s_dth[s + m - 2 + kPad]; }
#pragma unroll
            for (int m = 0; m < 5; ++m) {
                double v = mn[m] + sd * u[m];
                if (v < lo) v = lo;
                if (v > hi) v = hi;
                u[m] = v;
                if (kFuse) {
                    const double nz = v - th[m];
                    w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = nz;
                    double sacc = dt5[m];
                    sacc = fma(c1, w0, sacc); sacc = fma(c2, w1, sacc); sacc = fma(c3, w2, sacc); sacc = fma(c4, w3, sacc); sacc = fma(c5, w4, sacc);
                    ss = fma(sacc, sacc, ss);
                    double qs = r0 * w4;
                    qs = fma(r1, w3, qs); qs = fma(r2, w2, qs); qs = fma(r3, w1, qs); qs = fma(r4, w0, qs);
                    quad = fma(w4, qs, quad);
                }
            }
#pragma unroll
            for (int m = 0; m < 5; ++m) col[s + m] = u[m];
        }
        for (; s < b; ++s) {
            double theta;
            const double v = sample_of(s, col[s], theta);
            col[s] = v;
            if (kFuse) push(v - theta, s, owns(s), true);
        }
        if (kFuse) {
            if (!last) { push(hp0, b, owns(b), false); push(hp1, b + 1, owns(b + 1), false); }
            else {
#pragma unroll
                for (int j = 0; j < 5; ++j) push(0.0, T + j, owns(T + j), false);   // rows up to T + 2 = N - 4: zero noise
            }
        }
    }
    __syncthreads();
    if (kFuse) {
        s_part[warp * 32 + lane] = ss;
        s_part[128 + warp * 32 + lane] = quad;
    }
    __syncthreads();
    // ---- phase 3b: lane = time step; warp w writes rollouts 8 w .. 8 w + 7 of the tile ----
    {
        double* const proj = p.proj;
        const bool store_noise = p.noise_from_rollouts == 0;
        const int row_stride = D * T;                        // doubles between the rows of consecutive rollouts of one joint
        const int c_begin = warp * 8, c_end = min(c_begin + 8, ncol);
        double* out_v = p.rollouts + (((size_t)q * p.slots + (k0 + c_begin)) * D + d) * T;
        double* out_n = p.noise + (((size_t)q * p.slots + (k0 + c_begin)) * D + d) * T;
        const double* tile_row = s_tile + c_begin * S;
        // theta of this lane's time steps, once for all rows (T <= STOMP_B200_MAX_TIME_STEPS = 256: eight per lane)
        double th_reg[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) th_reg[j] = (lane + 32 * j < T) ? s_th[lane + 32 * j] : 0.0;
        for (int c = c_begin; c < c_end; ++c, out_v += row_stride, out_n += row_stride, tile_row += S) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int t = lane + 32 * j;
                if (t < T) {
                    const double v = tile_row[t];
                    out_v[t] = v;
                    if (store_noise) out_n[t] = v - th_reg[j];
                }
            }
            if (proj) {                                      // configurations with rollout reuse: computeProjectedNoise with M = I (PolicyImprovement.cpp:430-440)
                double* proj_row = proj + (((size_t)q * p.slots + (k0 + c)) * D + d) * T;
                for (int t = lane; t < T; t += 32) { const double th = th_all[kPad + t]; proj_row[t] = th + (tile_row[t] - th); }
            }
        }
    }
    if (warp == 0 && live) {
        const int k = k0 + lane;
        double* srow = p.sums + ((size_t)q * p.gslots + (p.gen_offset + k)) * p.sumw;
        if (kFuse) {
            const double sw = p.rule_sqrt_w[0];
            const double kappa = (p.dt * p.control_cost_weight) * (sw * sw);
            const double ss_all = (s_part[lane] + s_part[32 + lane]) + (s_part[64 + lane] + s_part[96 + lane]);
            const double quad_all = (s_part[128 + lane] + s_part[160 + lane]) + (s_part[192 + lane] + s_part[224 + lane]);
            store_row_sums(p, q, k, d, kappa * ss_all + edge_cost_sum(p, q, d), quad_all);   // rows_mask is 3 here
        }
        if (d == 0) {                   // S_k = sum_t state cost is accumulated with atomics by the state kernel: zeroed here
            srow[0] = 0.0;
            if (p.s_compact) p.s_compact[(size_t)q * p.gslots + (p.gen_offset + k)] = 0.0;
        }
    }
    tls.end();
}

// injected unit noise (parity mode): epilogue only
__global__ void __launch_bounds__(256)
shift_rollouts_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ JointLimits robot)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 0);
    const int per_query = p.num_gen * p.D * p.T;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < per_query; e += gridDim.x * blockDim.x) {
        const int t = e % p.T;
        const int kd = e / p.T;
        const int d = kd % p.D, k = kd / p.D;
        shift_clamp_store(p, robot, q, k, d, t, p.unit_noise[(size_t)q * per_query + e]);
    }
    tls.end();
}

// =====================================================================================================
// K4: state verdict — FK of the chain, sphere centres, SDF lookups
// (what robot_model does for OptimizationTask::computeCollisionCost, OptimizationTask.cpp:183-204)
// =====================================================================================================
template <bool kSimple, class JointValue>
__device__ __forceinline__ bool state_collides(const RobotParams& robot, const SdfParams& sdf, JointValue joint_value)
{
    Frame f;
    frame_identity(f);
    bool hit = false;
    const int nj = robot.num_joints;
    for (int d = 0; d < nj; ++d) {
        apply_joint<kSimple>(f, robot.joint[d], joint_value(d));
        const int s1 = robot.sphere_begin[d + 1];
        for (int s = robot.sphere_begin[d]; s < s1; ++s) {
            double cx, cy, cz;
            sphere_centre(f, robot.sphere[s], cx, cy, cz);
            const double dist = (double)__ldg(sdf.grid + sdf_index(sdf, cx, cy, cz));
            hit |= (dist - robot.sphere[s].r) < 0.0;
        }
    }
    return hit;
}

// K5 + K6: PolicyImprovement::computeRolloutControlCosts / computeRolloutCumulativeCosts
// (PolicyImprovement.cpp:442-495) and the n^T R n of the noise adaptation (:656-663) for the generated rollouts.
// One WARP per (rollout, joint) row.  The warp stages the padded trajectory x = theta + noise and the noise in
// its own shared-memory rows with coalesced loads (consecutive lanes, consecutive time steps), then every lane
// evaluates four consecutive elements from one 10-wide window read as five 16-byte loads — 2.5 KB of shared
// memory traffic per row instead of 7 KB for per-element windows, no block barrier, no address-divergent
// global load (an uncoalesced version of this loop saturates the L1 pipe, a shuffle version the SHFL pipe).
constexpr int kRowWarps = 8;
__host__ __device__ inline int control_row_x_stride(int N) { return 4 + ((N + 127) / 128) * 128 + 16; }   // even: every warp row stays 16-byte aligned
__host__ __device__ inline int control_row_n_stride(int T) { return ((T + 127) / 128) * 128 + 16; }

__global__ void __launch_bounds__(kRowWarps * 32)
control_rows_kernel(const __grid_constant__ LoopParams p)
{
    extern __shared__ __align__(16) double smem[];
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 6);
    const int T = p.T, D = p.D, N = p.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int XS = control_row_x_stride(N), NS = control_row_n_stride(T);
    double* xs = smem + (size_t)warp * (XS + NS);   // xs[3 + i] = x_all[i]; zeros on both sides
    double* ns = xs + XS;                           // ns[t] = noise[t]; zeros beyond T
    const int row = blockIdx.x * kRowWarps + warp;
    if (row < p.num_gen * D) {      // warp-uniform
        const int k = row / D, d = row - k * D;
        const double* nz = p.rows_noise + (((size_t)q * p.slots + k) * D + d) * T;
        const double* th = p.theta_all + ((size_t)q * D + d) * N;
        double* cc_out = p.control_costs ? p.control_costs + (((size_t)q * p.slots + k) * D + d) * T : nullptr;
        // ---- stage ----
        for (int i = lane; i < XS; i += 32) {
            const int j = i - 3;
            double v = 0.0;
            if (j >= 0 && j < N) {
                v = th[j];
                if (j >= kPad && j < kPad + T) v = v + nz[j - kPad];
            }
            xs[i] = v;
        }
        for (int t = lane; t < NS; t += 32) ns[t] = (t < T) ? nz[t] : 0.0;
        __syncwarp();
        // ---- control costs: lane handles elements i0 .. i0 + 3 of every 128-wide pass ----
        double C_part = 0.0, quad = 0.0;
        for (int base = 0; base < N; base += 128) {
            const int i0 = base + 4 * lane;
            double w[10];   // w[j] = x_all[i0 - 3 + j]
            const double2* src = reinterpret_cast<const double2*>(xs + i0);
#pragma unroll
            for (int j = 0; j < 5; ++j) { const double2 v = src[j]; w[2 * j] = v.x; w[2 * j + 1] = v.y; }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = i0 + e;
                if (i < N) {
                    const double cost = (p.st_uniform && i >= 3 && i < N - 3)
                                            ? interior_row_cost<0, 6>(p, [&](int o) { return w[e + o]; })
                                            : band_row_cost(p, i, [&](int j) { return xs[3 + j]; });
                    C_part += cost;
                    // per-timestep layout for read-backs; fold_control_costs_kernel adds the padding rows in the reference's order
                    if (cc_out && i >= kPad && i < kPad + T) cc_out[i - kPad] = cost;
                }
            }
        }
        // ---- n^T R n: sum_t n_t (R_tt n_t + 2 sum_{o>0} R_{t,t+o} n_{t+o}); the noise is zero outside [0, T) ----
        if (p.use_noise_adaptation) {
            for (int base = 0; base < T; base += 128) {
                const int t0 = base + 4 * lane;
                double m[10];   // m[j] = noise[t0 + j]
                const double2* src = reinterpret_cast<const double2*>(ns + t0);
#pragma unroll
                for (int j = 0; j < 5; ++j) { const double2 v = src[j]; m[2 * j] = v.x; m[2 * j + 1] = v.y; }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int t = t0 + e;
                    if (t < T) {
                        auto nt = [&](int o) { return m[e + o]; };
                        quad += p.r_toeplitz ? quad_term<kRBand>(p.r_diag, nt)
                                             : quad_term<kRBand>(p.Rband + (size_t)t * (2 * kRBand + 1) + kRBand, nt);
                    }
                }
            }
        }
        C_part = warp_sum(C_part);
        quad = warp_sum(quad);
        if (lane == 0) store_row_sums(p, q, k, d, C_part, quad);
    }
    tls.end();
}

// costs of the band-table rows i in {0, 1, 2, N-3, N-2, N-1} of the single active rule for every (query, joint):
// they read x_all[0..5] / x_all[N-6..N-1] only, i.e. the padding, which a solve never changes
// (CovariantMovementPrimitive::updateParameters touches the free block only, CovariantMovementPrimitive.cpp:476-479).
__global__ void edge_rows_kernel(const __grid_constant__ LoopParams p)
{
    const int q = blockIdx.x, N = p.N;
    for (int e = threadIdx.x; e < p.D * 6; e += blockDim.x) {
        const int d = e / 6, r = e - d * 6;
        const double* th = p.theta_all + ((size_t)q * p.D + d) * N;
        p.edge_cost[(size_t)q * p.D * 6 + e] = band_row_cost(p, r < 3 ? r : N - 6 + r, [&](int j) { return th[j]; });
    }
}

// The same rows for the common shape — one active differentiation rule (interior rows all carry the same 7
// taps), Toeplitz R, even T — without shared memory: lane l of the row's warp owns the padded indices
// i0 .. i0+3 (i0 = 4l) and loads the 12-wide ALIGNED windows theta_all[i0-4 .. i0+7] and noise[i0-10 .. i0+1]
// as six 16-byte loads each (a 16-byte pair is inside or outside the row as a whole, because T, N and
// TRAJECTORY_PADDING are even).  Everything a lane needs — the stencil windows of its four elements and the
// noise windows of its four n^T R n terms — is in those registers, so the row costs ~330 warp instructions
// instead of ~1300.  Rows 0..2 and N-3..N-1 (band-table rows) only touch the fixed padding; six lanes
// evaluate them from the table after the main pass.
// kTaps5: taps -3 and +3 are zero (the acceleration rule).  kRb4: R[t][t+5] = R[t][t+6] = 0 (follows from it).
template <bool kTaps5, bool kRb4>
__global__ void __launch_bounds__(256, 4)
control_rows_fast_kernel(const __grid_constant__ LoopParams p)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 6);
    const int T = p.T, D = p.D, N = p.N;
    const int lane = threadIdx.x & 31;
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row < p.num_gen * D) {      // warp-uniform
        const int k = row / D, d = row - k * D;
        const double* nz = p.rows_noise + (((size_t)q * p.slots + k) * D + d) * T;
        const double* th = p.theta_all + ((size_t)q * D + d) * N;
        double* cc_out = p.control_costs ? p.control_costs + (((size_t)q * p.slots + k) * D + d) * T : nullptr;
        constexpr int kNoisePairs = kRb4 ? 6 : 7;
        constexpr int kBand = kRb4 ? 4 : kRBand;
        double C_part = 0.0, quad = 0.0;
        // band-table rows 0..2 and N-3..N-1 only see the fixed padding: their costs are per (query, joint) constants
        // of the solve (edge_rows_kernel); six lanes pick them up and add them before the warp sum (not edge_cost_sum: that
        // order of the additions is this kernel's own)
        const double edge = (lane < 6) ? p.edge_cost[((size_t)q * D + d) * 6 + lane] : 0.0;
        for (int base = 0; base < N; base += 128) {
            const int i0 = base + 4 * lane;
            if (i0 >= N) continue;
            double W[12];             // W[j] = theta_all[i0 - 4 + j], then x_all
            double M[2 * kNoisePairs];   // M[j] = noise[i0 - 10 + j], zero outside [0, T)
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const int idx = i0 - 4 + 2 * j;
                double2 v = make_double2(0.0, 0.0);
                if (idx >= 0 && idx < N) v = *reinterpret_cast<const double2*>(th + idx);
                W[2 * j] = v.x; W[2 * j + 1] = v.y;
            }
#pragma unroll
            for (int j = 0; j < kNoisePairs; ++j) {
                const int idx = i0 - 10 + 2 * j;
                double2 v = make_double2(0.0, 0.0);
                if (idx >= 0 && idx < T) v = *reinterpret_cast<const double2*>(nz + idx);
                M[2 * j] = v.x; M[2 * j + 1] = v.y;
            }
            // x_all = theta_all + noise on the free block (adding the zero outside it leaves theta_all)
#pragma unroll
            for (int j = 0; j < 12; ++j) W[j] = W[j] + M[j];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = i0 + e;
                const double cost = interior_row_cost<kTaps5 ? 1 : 0, kTaps5 ? 5 : 6>(p, [&](int o) { return W[e + o + 1]; });
                if (i >= 3 && i < N - 3) {
                    C_part += cost;
                    // per-timestep layout for read-backs; fold_control_costs_kernel adds the padding rows in the reference's order
                    if (cc_out && i >= kPad && i < kPad + T) cc_out[i - kPad] = cost;
                }
            }
            // n^T R n terms of t = i - kPad: n_t (R_tt n_t + 2 sum_{o>0} R_{t,t+o} n_{t+o}), n_t = M[e + 4]
            if (p.use_noise_adaptation) {
#pragma unroll
                for (int e = 0; e < 4; ++e) quad += quad_term<kBand>(p.r_diag, [&](int o) { return M[e + 4 + o]; });   // zero noise outside [0, T): no guard needed
            }
        }
        C_part += edge;
        C_part = warp_sum(C_part);
        quad = warp_sum(quad);
        if (lane == 0) store_row_sums(p, q, k, d, C_part, quad);
    }
    tls.end();
}

// The rows once more, for the shipped shape of the operator (one rule whose interior taps are -2..+2 — the
// acceleration rule — hence R five-banded and Toeplitz; even T): the leanest form.  A warp owns EIGHT consecutive
// (rollout, joint) rows — 8 T contiguous doubles of `noise` — and copies them once, with coalesced 16-byte loads,
// into zero-padded shared-memory rows; then lane (r, kq) walks quarter kq of row r SEQUENTIALLY with the stencil
// and noise windows sliding through registers (fully unrolled: no register moves), four elements per pair of
// 16-byte shared loads.  No bounds test inside the walk (the padding is zeros and the band-table rows come from
// edge_cost), a two-step shuffle per row instead of five: ~120 warp instructions per row, ~85 % of them FP64
// arithmetic, against ~510 for control_rows_fast_kernel.
// Row strides are == 2 (mod 16) doubles: the 16-byte loads of a quarter-warp (2 rows x 4 quarters) hit 32
// distinct banks.  kGroups = groups of four elements per lane = ceil(N / 16).
// One warp per CTA: 8.3 KB of shared memory and 76 registers let 26 such CTAs live on an SM, so the 24.2 tiles per
// SM of BASELINE config 3 (28672 rows / 8 / 148) run as ONE wave; with 8-warp CTAs (3 per SM = 24 warps) the
// 25th tile of an SM waited for a whole CTA and doubled the kernel's time (profiles/r1q).
constexpr int kTileWarps = 1;
__host__ __device__ constexpr int tile_groups(int N) { return (N + 15) / 16; }
__host__ __device__ constexpr int tile_noise_stride(int groups) { return ((16 * groups + 14 - 2 + 15) / 16) * 16 + 2; }   // >= 16 groups + 14

template <int kGroups, bool kStore>
__global__ void __launch_bounds__(kTileWarps * 32, 26)
control_rows_tile_kernel(const __grid_constant__ LoopParams p)
{
    extern __shared__ __align__(16) double smem[];
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 6);
    const int T = p.T, D = p.D, N = p.N;
    constexpr int E = 4 * kGroups;                    // elements per lane
    constexpr int NS = tile_noise_stride(kGroups);    // ns[r][8 + t] = noise[t]; zeros elsewhere
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* ns = smem + (size_t)warp * 8 * NS;
    const int nrows = p.num_gen * D;
    const int c0 = (blockIdx.x * kTileWarps + warp) * 8;      // first row of this warp

    if (c0 < nrows) {
        // ---- stage: rows c0 .. c0+7 are contiguous in `noise` ----
        const double* src = p.rows_noise + ((size_t)q * p.slots * D + c0) * T;
        // cp.async (16 bytes, zero-filled outside the row): all ~24 copies of a lane are in flight at once.  As a
        // load-then-store loop the compiler kept one load in flight per lane and the stage alone cost 24 L2 round trips,
        // ~6 us of a tile's ~10 us (profiles/r1u: long-scoreboard stalls on the eight STS.128).
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const bool row_ok = c0 + r < nrows;
#pragma unroll
            for (int j0 = 0; j0 < NS; j0 += 64) {
                const int j = j0 + 2 * lane;
                if (j < NS) {
                    const int t = j - 8;
                    const bool in = row_ok && t >= 0 && t < T;
                    const double* g = in ? src + (size_t)r * T + t : src;
                    const unsigned dst = (unsigned)__cvta_generic_to_shared(ns + r * NS + j);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(dst), "l"(g), "r"(in ? 16 : 0) : "memory");
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncwarp();
    const int r = lane >> 2, kq = lane & 3;
    const int c = c0 + r;
    if (c0 < nrows) {          // warp-uniform
        const bool live = c < nrows;
        const int k = live ? c / D : 0, d = live ? c - k * D : 0;
        const double edge = (live && kq == 0) ? edge_cost_sum(p, q, d) : 0.0;
        const int i_begin = kq * E;
        const double* nrow = ns + r * NS + i_begin;          // nrow[m] = noise[i_begin + m - 8]
        const double* trow = p.theta_all + ((size_t)q * D + d) * N + i_begin - 2;   // trow[m] = theta_all[i_begin + m - 2] (L1-resident)
        // 16-byte pair of theta_all at trow[m], zeros outside the row (only masked elements look there)
        auto theta_pair = [&](int m) {
            const int j = i_begin - 2 + m;
            return (j >= 0 && j < N) ? *reinterpret_cast<const double2*>(trow + m) : make_double2(0.0, 0.0);
        };
        double* cc_out = (kStore && live) ? p.control_costs + (((size_t)q * p.slots + k) * D + d) * T : nullptr;
        // windows for the group at i: nw[m] = noise[i - 8 + m], m < 10 ; xw[m] = x_all[i - 2 + m], m < 8
        double nw[10], xw[8];
#pragma unroll
        for (int m = 0; m < 6; m += 2) { const double2 v = *reinterpret_cast<const double2*>(nrow + m); nw[m + 4] = v.x; nw[m + 5] = v.y; }
#pragma unroll
        for (int m = 0; m < 4; m += 2) {
            const double2 v = theta_pair(m);
            xw[m + 4] = v.x + nw[m + 4]; xw[m + 5] = v.y + nw[m + 5];
        }
        double C0 = 0.0, C1 = 0.0, Q0 = 0.0, Q1 = 0.0;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const int i = i_begin + 4 * g;
            // slide: four new noise values and four new x values
#pragma unroll
            for (int m = 0; m < 6; ++m) nw[m] = nw[m + 4];
#pragma unroll
            for (int m = 0; m < 4; ++m) xw[m] = xw[m + 4];
            {
                const double2 a = *reinterpret_cast<const double2*>(nrow + 4 * g + 6), b = *reinterpret_cast<const double2*>(nrow + 4 * g + 8);
                nw[6] = a.x; nw[7] = a.y; nw[8] = b.x; nw[9] = b.y;
                const double2 ta = theta_pair(4 * g + 4), tb = theta_pair(4 * g + 6);
                // x_all[j] = theta_all[j] + noise[j - 6]: j = i + 2 + m  <->  nw[4 + m]
                xw[4] = ta.x + nw[4]; xw[5] = ta.y + nw[5]; xw[6] = tb.x + nw[6]; xw[7] = tb.y + nw[7];
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                // element i + e: taps -2 .. +2 on x_all
                double cost = interior_row_cost<1, 5>(p, [&](int o) { return xw[e + o - 1]; });
                if ((unsigned)(i + e - 3) >= (unsigned)(N - 6)) cost = 0.0;     // band-table rows and the zero padding beyond N
                if (e & 1) C1 += cost; else C0 += cost;
                if (kStore && cc_out && i + e >= kPad && i + e < kPad + T) cc_out[i + e - kPad] = cost;
                // n^T R n term of t = i + e - 6: n_t = nw[2 + e]; zero outside [0, T), no guard needed
                const double term = quad_term<4>(p.r_diag, [&](int o) { return nw[2 + e + o]; });
                if (e & 1) Q1 += term; else Q0 += term;
            }
        }
        double C_part = (C0 + C1) + edge, quad = Q0 + Q1;
        C_part += __shfl_xor_sync(0xffffffffu, C_part, 1); quad += __shfl_xor_sync(0xffffffffu, quad, 1);
        C_part += __shfl_xor_sync(0xffffffffu, C_part, 2); quad += __shfl_xor_sync(0xffffffffu, quad, 2);
        if (live && kq == 0) store_row_sums(p, q, k, d, C_part, quad);
    }
    tls.end();
}

// fold of the padding rows into the first / last free step in the reference's order, for the stored
// per-timestep control costs (read-backs only; one thread per row)
__global__ void __launch_bounds__(128)
fold_control_costs_kernel(const __grid_constant__ LoopParams p)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q) || !p.control_costs) return;
    const int T = p.T, D = p.D, N = p.N;
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= p.num_gen * D) return;
    const int k = row / D, d = row - k * D;
    const double* nz = p.rows_noise + (((size_t)q * p.slots + k) * D + d) * T;
    const double* th = p.theta_all + ((size_t)q * D + d) * N;
    double* cc = p.control_costs + (((size_t)q * p.slots + k) * D + d) * T;
    auto xall = [&](int j) { return (j >= kPad && j < kPad + T) ? th[j] + nz[j - kPad] : th[j]; };
    double first = cc[0], last = cc[T - 1];
    for (int i = 0; i < kPad; ++i) { first += band_row_cost(p, i, xall); last += band_row_cost(p, N - (i + 1), xall); }
    cc[0] = first;
    cc[T - 1] = last;
}

// K4: Stomp::doExecuteRollouts (stomp/src/Stomp.cpp:206-229) -> Task::execute for every generated rollout:
// one thread per (rollout, timestep) state, noisy parameters read coalesced along t, FK in registers, SDF
// gathers through the read-only path, cost / verdict written back; S_k = sum_t cost accumulated with
// atomicAdd (the terms are 0 / 1, so the double sum is exact in any order).  This is the roofline kernel:
// 8D + 4S + 9 algorithmic bytes per state.
// It serves every world-only state pass the generated kernel cannot (no NVRTC, STOMP_B200_STATES=generic, joint values
// that kernel cannot vouch for); null pointers in StateKernelArgs as in states_self_collision_kernel, no NoiselessTail.
template <bool kSimple>
__global__ void __launch_bounds__(128)
rollout_states_kernel(const __grid_constant__ StateKernelArgs a, const __grid_constant__ RobotParams robot,
                      const __grid_constant__ SdfParams sdf)
{
    const int q = blockIdx.y;
    if (a.tile_counter && blockIdx.x == 0 && q == 0 && threadIdx.x < 4) a.tile_counter[threadIdx.x] = 0u;   // for the next sampling launch
    if (a.honour_stop && a.stop[q] != 0) return;
    TimelineScope tls(a.timeline);
    const SdfParams field = query_field(a.query_sdf, q, sdf);     // the field of this query's scene
    const int T = a.T;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < a.num_gen * T) {
        const int k = idx / T, t = idx - k * T;
        const double* xq = a.rollouts + ((size_t)q * a.slots + k) * a.rollout_stride + t;
        const size_t rs = (size_t)a.row_stride;
        const bool hit = state_collides<kSimple>(robot, field, [&](int d) { return xq[(size_t)d * rs]; });
        const size_t o = ((size_t)q * a.slots + k) * T + t;
        if (a.state_costs) a.state_costs[o] = hit ? 1.0 : 0.0;
        if (a.verdicts) a.verdicts[o] = hit ? 1 : 0;
        if (a.validity && t == T - 1) a.validity[(size_t)q * a.slots + k] = hit ? 0 : 1;   // last timestep only (OptimizationTask.cpp:192-202)
        if (hit && a.sums) atomicAdd(a.sums + ((size_t)q * a.gslots + (a.gen_offset + k)) * a.sumw, 1.0);
        if (hit && a.s_compact) atomicAdd(a.s_compact + (size_t)q * a.gslots + (a.gen_offset + k), 1.0);
    }
    tls.end();
}

// -----------------------------------------------------------------------------------------------------
// Alternative state costs (SURVEY.md 8f rank 4; both off in the shipped configuration, stomp_b200_set_cost_extras):
//   smooth obstacle cost: weight * sum_s max(0, (r_s + margin) - d_s) over the link spheres in index order, in place of
//     the 0 / 1 verdict cost — the non-boolean obstacle shape of stomp/test/stomp_2d_test.cpp:337-363 for spheres and a
//     distance field;
//   joint-constraint cost: OptimizationTask::computeJointsConstraintCost / getConstrainDifference
//     (src/wrappers/stomp/OptimizationTask.cpp:206-237; the call at :169-172 is commented out in the reference):
//     + weight * sum_d max(0, |value_d - q_d| - tolerance_d).
// They run as a pass of their own after the state kernel (generic FK; the verdicts stay the state kernel's), followed by
// a fixed-order row sum for S_k — costs are no longer small integers, so the state kernel's atomic count does not serve.
// -----------------------------------------------------------------------------------------------------
struct CostExtras {
    int32_t smooth, joint_constraint;
    double smooth_margin, smooth_weight, jc_weight;
    double jc_value[STOMP_B200_MAX_DIMS], jc_tolerance[STOMP_B200_MAX_DIMS];
};

template <class JointValue>
__device__ __forceinline__ double extra_state_cost(const RobotParams& robot, const SdfParams& sdf, const CostExtras& x,
                                                   JointValue joint_value, double binary_cost)
{
    double cost = binary_cost;
    if (x.smooth) {
        Frame f;
        frame_identity(f);
        double pen = 0.0;
        for (int d = 0; d < robot.num_joints; ++d) {
            apply_joint<false>(f, robot.joint[d], joint_value(d));
            for (int s = robot.sphere_begin[d]; s < robot.sphere_begin[d + 1]; ++s) {
                double cx, cy, cz;
                sphere_centre(f, robot.sphere[s], cx, cy, cz);
                const double soft = robot.sphere[s].r + x.smooth_margin;
                const double depth = soft - (double)__ldg(sdf.grid + sdf_index(sdf, cx, cy, cz));
                if (depth > 0.0) pen = pen + depth;
            }
        }
        cost = x.smooth_weight * pen;
    }
    if (x.joint_constraint) {
        double cc = 0.0;
        for (int d = 0; d < robot.num_joints; ++d) {
            const double diff = x.jc_tolerance[d] - fabs(x.jc_value[d] - joint_value(d));
            if (diff < 0.0) cc = cc + (-1.0 * diff);
        }
        cost = cost + x.jc_weight * cc;
    }
    return cost;
}

// rewrites state_costs of the generated rollouts; thread per (rollout, time step)
__global__ void __launch_bounds__(128)
state_cost_extras_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ RobotParams robot,
                         const __grid_constant__ SdfParams sdf, const __grid_constant__ CostExtras x)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.num_gen * T) return;
    const int k = idx / T, t = idx - k * T;
    const double* xq = p.rollouts + ((size_t)q * p.slots + k) * D * T + t;
    const size_t o = ((size_t)q * p.slots + k) * T + t;
    const SdfParams field = query_field(p.query_sdf, q, sdf);
    p.state_costs[o] = extra_state_cost(robot, field, x, [&](int d) { return xq[(size_t)d * T]; }, p.state_costs[o]);
}

// S_k = sum_t state_costs[k][t] of the generated rollouts, one warp per rollout, fixed order
__global__ void __launch_bounds__(256)
state_row_sums_kernel(const __grid_constant__ LoopParams p)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= p.num_gen) return;
    const double* row = p.state_costs + ((size_t)q * p.slots + k) * p.T;
    double s = 0.0;
    for (int t = lane; t < p.T; t += 32) s += row[t];
    s = warp_sum(s);
    if (lane == 0) {
        p.sums[((size_t)q * p.gslots + (p.gen_offset + k)) * p.sumw] = s;
        if (p.s_compact) p.s_compact[(size_t)q * p.gslots + (p.gen_offset + k)] = s;
    }
}

// the same pass for stomp_b200_evaluate_states: theta [K][D][Tq], costs [K][Tq]
__global__ void __launch_bounds__(128)
evaluate_extras_kernel(const __grid_constant__ RobotParams robot, const __grid_constant__ SdfParams sdf, const __grid_constant__ CostExtras x,
                       const double* __restrict__ theta, int K, int Tq, double* __restrict__ costs)
{
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)K * Tq) return;
    const int k = (int)(idx / Tq), t = (int)(idx - (size_t)k * Tq);
    const double* base = theta + (size_t)k * robot.num_joints * Tq + t;
    costs[idx] = extra_state_cost(robot, sdf, x, [&](int d) { return base[(size_t)d * Tq]; }, costs[idx]);
}

// the noise-less rollout record written out as the regular rollout slot the reference appends
// (PolicyImprovement.cpp:304-308): parameters = the current policy parameters, zero noise, the recorded costs.
// Called by one CTA of rollout_weights_kernel (before the update changes the parameters); the loop itself
// reads the record, the slot serves rollout reuse and read-backs.
__device__ __forceinline__ void materialise_noiseless(const LoopParams& p, int q, int tid, int nthreads)
{
    const int T = p.T, D = p.D, N = p.N, k = p.noiseless_slot;
    for (int e = tid; e < D * T; e += nthreads) {
        const int d = e / T, t = e - d * T;
        const double th = p.theta_all[((size_t)q * D + d) * N + kPad + t];
        const size_t o = (((size_t)q * p.slots + k) * D) * T + e;
        p.rollouts[o] = th;
        p.noise[o] = 0.0;
        if (p.noise_proj) p.noise_proj[o] = 0.0;
        if (p.proj) p.proj[o] = th;
        if (p.control_costs) p.control_costs[o] = p.nl_control[(size_t)q * D * T + e];
    }
    for (int t = tid; t < T; t += nthreads) {
        p.state_costs[((size_t)q * p.slots + k) * T + t] = p.nl_state[(size_t)q * T + t];
        p.verdicts[((size_t)q * p.slots + k) * T + t] = p.nl_verdict[(size_t)q * T + t];
    }
    for (int e = tid; e < p.sumw; e += nthreads)
        p.sums[((size_t)q * p.gslots + p.noiseless_gslot) * p.sumw + e] = p.nl_sums[(size_t)q * p.sumw + e];
}

// =====================================================================================================
// Self collision (SURVEY.md §8f rank 3: the "self" half of robot_model's isStateValid, with the SRDF's disabled
// link pairs removed on the host — reference test/data/kuka_iiwa.srdf:46-70).  A state is in collision when a
// link sphere is inside an obstacle (as above) OR two spheres of a listed pair overlap:
//   |c_i - c_j|^2 < (r_i + r_j)^2,   |.|^2 = fma(dz, dz, fma(dy, dy, dx * dx)),   the limit squared on the host.
// While a pair list is set, this kernel or the generated one with the pair rule serves every state pass in place of
// the world-only kernels (engine.cu: launch_state_pass).  It takes the same StateKernelArgs, so the noisy rollouts,
// the padded policy rows of the noise-less rollout and stomp_b200_evaluate_states all go through it.
// Sphere centres and one bounding sphere per link live in thread-local memory (L1).  The host sorts the pairs into
// blocks by link pair; a block is only walked when the two links' bounding spheres overlap.  The bounding radii are
// inflated by far more than the rounding of the centres, so the cull never removes a pair that the exact rule
// accepts: verdicts stay those of the plain list walk (what the oracle does).  Measured on the dual-arm workload
// (K=2048, T=150, 560 pairs): 635 us as a plain list walk.
// =====================================================================================================
// struct SelfPairs: kinematics.cuh (the run-time specialised kernel with the pair rule takes it too)

template <int kSphereCapacity, bool kSimple>   // thread-local centre storage sized by the host to the robot (32 / 64 / 128)
__global__ void __launch_bounds__(128)
states_self_collision_kernel(const __grid_constant__ StateKernelArgs a, const __grid_constant__ RobotParams robot,
                             const __grid_constant__ SdfParams sdf, const __grid_constant__ SelfPairs pairs)
{
    const int q = blockIdx.y;
    if (a.tile_counter && blockIdx.x == 0 && q == 0 && threadIdx.x < 4) a.tile_counter[threadIdx.x] = 0u;
    if (a.honour_stop && a.stop[q] != 0) return;
    if (a.timeline && threadIdx.x == 0) {
        unsigned long long t0;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
        atomicMin(a.timeline, t0);
    }
    const SdfParams field = query_field(a.query_sdf, q, sdf);     // the field of this query's scene
    const int T = a.T;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < a.num_gen * T) {
        const int k = idx / T, t = idx - k * T;
        const double* xq = a.rollouts + ((size_t)q * a.slots + k) * a.rollout_stride + t;
        const size_t rs = (size_t)a.row_stride;
        double c[3 * kSphereCapacity];
        double bc[3 * STOMP_B200_MAX_DIMS];
        Frame f;
        frame_identity(f);
        bool hit = false;
        const int nj = robot.num_joints;
        for (int d = 0; d < nj; ++d) {
            apply_joint<kSimple>(f, robot.joint[d], xq[(size_t)d * rs]);
            const double bx = __ldg(pairs.link_bound + 4 * d), by = __ldg(pairs.link_bound + 4 * d + 1), bz = __ldg(pairs.link_bound + 4 * d + 2);
            bc[3 * d] = fma(f.r02, bz, fma(f.r01, by, fma(f.r00, bx, f.px)));
            bc[3 * d + 1] = fma(f.r12, bz, fma(f.r11, by, fma(f.r10, bx, f.py)));
            bc[3 * d + 2] = fma(f.r22, bz, fma(f.r21, by, fma(f.r20, bx, f.pz)));
            const int s1 = robot.sphere_begin[d + 1];
            for (int s = robot.sphere_begin[d]; s < s1; ++s) {
                double cx, cy, cz;
                sphere_centre(f, robot.sphere[s], cx, cy, cz);
                c[3 * s] = cx; c[3 * s + 1] = cy; c[3 * s + 2] = cz;
                const double dist = (double)__ldg(field.grid + sdf_index(field, cx, cy, cz));
                hit |= (dist - robot.sphere[s].r) < 0.0;
            }
        }
        for (int b = 0; b < pairs.nblocks && !hit; ++b) {
            const int4 blk = __ldg(pairs.block + b);
            const double ex = bc[3 * blk.x] - bc[3 * blk.y];
            const double ey = bc[3 * blk.x + 1] - bc[3 * blk.y + 1];
            const double ez = bc[3 * blk.x + 2] - bc[3 * blk.y + 2];
            if (!(fma(ez, ez, fma(ey, ey, ex * ex)) < __ldg(pairs.block_limit2 + b))) continue;   // links too far apart
            for (int pr = blk.z; pr < blk.w; ++pr) {
                const int2 ij = __ldg(pairs.ij + pr);
                const double dx = c[3 * ij.x] - c[3 * ij.y];
                const double dy = c[3 * ij.x + 1] - c[3 * ij.y + 1];
                const double dz = c[3 * ij.x + 2] - c[3 * ij.y + 2];
                const double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
                if (d2 < __ldg(pairs.limit2 + pr)) { hit = true; break; }
            }
        }
        const size_t o = ((size_t)q * a.slots + k) * T + t;
        if (a.state_costs) a.state_costs[o] = hit ? 1.0 : 0.0;
        if (a.verdicts) a.verdicts[o] = hit ? 1 : 0;
        if (a.validity && t == T - 1) a.validity[(size_t)q * a.slots + k] = hit ? 0 : 1;
        if (hit && a.sums) atomicAdd(a.sums + ((size_t)q * a.gslots + (a.gen_offset + k)) * a.sumw, 1.0);
        if (hit && a.s_compact) atomicAdd(a.s_compact + (size_t)q * a.gslots + (a.gen_offset + k), 1.0);
    }
    if (a.timeline) {
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long t1;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
            atomicMax(a.timeline + 1, t1);
        }
    }
}

__global__ void sphere_centres_kernel(const __grid_constant__ RobotParams robot, const double* __restrict__ q, int n,
                                      double* __restrict__ centres)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Frame f;
    frame_identity(f);
    for (int d = 0; d < robot.num_joints; ++d) {
        apply_joint<false>(f, robot.joint[d], q[(size_t)i * robot.num_joints + d]);
        for (int s = robot.sphere_begin[d]; s < robot.sphere_begin[d + 1]; ++s) {
            double cx, cy, cz;
            sphere_centre(f, robot.sphere[s], cx, cy, cz);
            double* o = centres + ((size_t)i * robot.num_spheres + s) * 3;
            o[0] = cx; o[1] = cy; o[2] = cz;
        }
    }
}

// =====================================================================================================
// Reused rollouts (PolicyImprovement.cpp:188-255): control costs are recomputed for ALL rollouts every
// iteration (computeRolloutControlCosts, :442-449) on parameters_ + noise_projected_ with the new
// parameters.  One warp per (slot, joint) over the reused slots [first, first + count).
// =====================================================================================================
__global__ void __launch_bounds__(256)
reused_control_cost_kernel(const __grid_constant__ LoopParams p, int first, int count)
{
    extern __shared__ double smem[];
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D, N = p.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    double* x = smem + (size_t)warp * (N + T);
    double* stc = x + N;
    for (int task = blockIdx.x * nwarps + warp; task < count * D; task += gridDim.x * nwarps) {
        const int r = task / D, d = task - r * D, k = first + r;
        // control costs see parameters_ + noise_projected_ (PolicyImprovement.cpp:812-817), the quadratic form noise_
        const double* cc_noise = p.noise_proj ? p.noise_proj : p.noise;
        for (int i = lane; i < N; i += 32) {
            const double th = p.theta_all[((size_t)q * D + d) * N + i];
            double v = th;
            if (i >= kPad && i < kPad + T) v = th + cc_noise[(((size_t)q * p.slots + k) * D + d) * T + (i - kPad)];
            x[i] = v;
        }
        for (int t = lane; t < T; t += 32) stc[t] = p.state_costs[((size_t)q * p.slots + k) * T + t];
        __syncwarp();
        double C_d, cum_d;
        control_cost_sums(p, x, stc, lane, C_d, cum_d);
        if (p.control_costs) control_cost_store(p, x, lane, p.control_costs + (((size_t)q * p.slots + k) * D + d) * T);
        double s = 0.0;
        for (int t = lane; t < T; t += 32) s += stc[t];
        s = warp_sum(s);
        double quad = 0.0;
        if (p.use_noise_adaptation) {
            if (p.noise_proj) {      // x held parameters + M * noise: rebuild it with the unprojected noise
                __syncwarp();
                for (int t = lane; t < T; t += 32)
                    x[kPad + t] = p.theta_all[((size_t)q * D + d) * N + kPad + t] + p.noise[(((size_t)q * p.slots + k) * D + d) * T + t];
            }
            // x becomes the noise x - theta with a zero tail, in place
            const double* theta_row = p.theta_all + ((size_t)q * D + d) * N;
            __syncwarp();
            for (int t = lane; t < T + kPad; t += 32) x[kPad + t] = (t < T) ? x[kPad + t] - theta_row[kPad + t] : 0.0;
            __syncwarp();
            const double* n = x + kPad;
            for (int t = lane; t < T; t += 32) {
                auto nt = [&](int o) { return n[t + o]; };
                quad += p.r_toeplitz ? quad_term<kRBand>(p.r_diag, nt)
                                     : quad_term<kRBand>(p.Rband + (size_t)t * (2 * kRBand + 1) + kRBand, nt);
            }
            quad = warp_sum(quad);
        }
        if (lane == 0) {
            double* o = p.sums + ((size_t)q * p.gslots + k) * p.sumw;
            o[0] = s;
            o[1 + d] = C_d;
            o[1 + D + d] = cum_d;
            o[1 + 2 * D + d] = quad;
        }
        __syncwarp();
    }
}

// importance weights of the previous rollouts, rank by (-w, index), gather the best `reused` ones behind
// the generated block of the other buffer set and re-base their noise on the new parameters
// (PolicyImprovement.cpp:188-255).  One CTA per query.
struct ReuseParams {
    int32_t prev, reused, gen;
    const double* src_proj; const double* src_state; const uint8_t* src_verdict; const double* src_total;
    int32_t* order;           // [Q][slots] scratch
};
__global__ void __launch_bounds__(256)
reuse_rollouts_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ ReuseParams rp)
{
    __shared__ double scratch[32];
    extern __shared__ double w[];      // [prev]
    const int q = blockIdx.x;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D, N = p.N, tid = threadIdx.x;
    const double* total = rp.src_total + (size_t)q * p.gslots;
    double mn = 1e300, mx = -1e300;
    for (int r = tid; r < rp.prev; r += blockDim.x) { mn = fmin(mn, total[r]); mx = fmax(mx, total[r]); }
    mn = block_reduce<1>(mn, scratch);
    mx = block_reduce<2>(mx, scratch);
    double den = mx - mn;
    if (den < 1e-8) den = 1e-8;
    for (int r = tid; r < rp.prev; r += blockDim.x) w[r] = -exp(((-p.cost_scaling_h) * (total[r] - mn)) / den);
    __syncthreads();
    int32_t* order = rp.order + (size_t)q * p.slots;
    for (int r = tid; r < rp.prev; r += blockDim.x) {
        int rank = 0;
        const double wr = w[r];
        for (int s = 0; s < rp.prev; ++s) rank += (w[s] < wr) || (w[s] == wr && s < r);
        if (rank < rp.reused) order[rank] = r;
    }
    __syncthreads();
    for (int e = tid; e < rp.reused * D * T; e += blockDim.x) {
        const int t = e % T;
        const int rd = e / T;
        const int d = rd % D, r = rd / D;
        const int src = order[r], dst = rp.gen + r;
        const double* pjrow = rp.src_proj + (((size_t)q * p.slots + src) * D + d) * T;
        const double* throw_ = p.theta_all + ((size_t)q * D + d) * N + kPad;
        const double pj = pjrow[t];
        const double th = throw_[t];
        double nz = pj - th;                 // noise_projected_ = parameters_noise_projected_ - parameters_ (:201-203)
        const size_t o = (((size_t)q * p.slots + dst) * D + d) * T + t;
        p.proj[o] = pj;
        if (p.Minv) {                        // noise_ = inv_projection_matrix_ * noise_projected_ (:204)
            p.noise_proj[o] = nz;
            const double* mi = p.Minv + (size_t)t * T;
            double acc = 0.0;
            for (int j = 0; j < T; ++j) acc += mi[j] * (pjrow[j] - throw_[j]);
            nz = acc;
        }
        p.noise[o] = nz;
        p.rollouts[o] = th + nz;
    }
    for (int e = tid; e < rp.reused * T; e += blockDim.x) {
        const int t = e % T, r = e / T;
        const int src = order[r], dst = rp.gen + r;
        p.state_costs[((size_t)q * p.slots + dst) * T + t] = rp.src_state[((size_t)q * p.slots + src) * T + t];
        p.verdicts[((size_t)q * p.slots + dst) * T + t] = rp.src_verdict[((size_t)q * p.slots + src) * T + t];
    }
}

// =====================================================================================================
// K7: PolicyImprovement::computeRolloutProbabilities (PolicyImprovement.cpp:497-582), cumulative-cost mode:
// cumulative_costs_[d] is constant over t (:480), so one probability per (rollout, joint).
// One CTA of 1024 threads per (joint, query): min / max, exp + sum, normalise — three passes over K' cost rows
// that stay in L1.  The noise-less rollout is read from its record (and written out as a slot by the d == 0 CTA).
// =====================================================================================================
__device__ __forceinline__ const double* cost_row(const LoopParams& p, int q, int k)
{
    return (k == p.noiseless_gslot) ? p.nl_sums + (size_t)q * p.sumw : p.sums + ((size_t)q * p.gslots + k) * p.sumw;
}

// total_cost_ (PolicyImprovement.cpp:451-462) of global slot g from its cost row s = cost_row(p, q, g): the state costs
// plus the control costs of the D joints.  s and D are the caller's: read again after the caller's stores, they would
// be loads of their own.
__device__ __forceinline__ void store_total_cost(const LoopParams& p, int q, int g, const double* s, int D)
{
    double cost = s[0];
    for (int dd = 0; dd < D; ++dd) cost += s[1 + dd];
    p.total_cost[(size_t)q * p.gslots + g] = cost;
}

// grid (wblocks, D, Q), 512 threads.  Every CTA scans all K' rows for the min / max of its joint (two 8-byte loads per
// row, unrolled so that they are all in flight at once: this kernel is pure L2 latency), then weighs its own slice of
// the rollouts and leaves the sum of its unnormalised weights in wpart[block]; the consumers (weighted_update_kernel,
// read-backs) divide by the sum of the wblocks partials taken in block order.  wblocks <= 8 keeps the redundant scans
// cheap; one CTA per joint (tried) serialises eight L2 round trips and takes twice as long.
constexpr int kWeightThreads = 512;
constexpr int kWeightBlocksMax = 8;
__global__ void __launch_bounds__(kWeightThreads)
rollout_weights_kernel(const __grid_constant__ LoopParams p)
{
    __shared__ double scratch[32];
    const int d = blockIdx.y, q = blockIdx.z;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 2);
    const int D = p.D, n = p.num_rollouts, tid = threadIdx.x;
    double* prob = p.prob + (size_t)q * p.gslots * D;
    double* fprob = p.fprob + (size_t)q * p.gslots * D;
    const double h = p.cost_scaling_h;
    if (blockIdx.x == 0 && d == 0 && p.noiseless_slot >= 0) materialise_noiseless(p, q, tid, blockDim.x);

    double mn = 1e300, mx = -1e300;
#pragma unroll 8
    for (int k = tid; k < n; k += kWeightThreads) {
        const double* s = cost_row(p, q, k);
        const double cum = 1.0 * (s[0] + s[1 + d]);   // sum_t (state + control_d) as S + C_d; equals full_costs_[d]
        mn = fmin(mn, cum); mx = fmax(mx, cum);
    }
    mn = block_reduce<1>(mn, scratch); mx = block_reduce<2>(mx, scratch);
    double den = mx - mn;
    if (den < 1e-8) den = 1e-8;

    const int per_block = (n + gridDim.x - 1) / gridDim.x;
    const int k_end = min(n, (int)(blockIdx.x + 1) * per_block);
    double psum = 0.0;
#pragma unroll 2
    for (int k = blockIdx.x * per_block + tid; k < k_end; k += kWeightThreads) {
        const double* s = cost_row(p, q, k);
        // cumulative_costs_[d] and full_costs_[d] are the same number in this build (S + C_d), hence one weight
        const double pr = 1.0 * exp(((-h) * (1.0 * (s[0] + s[1 + d]) - mn)) / den);      // importance_weight_ = 1
        prob[(size_t)k * D + d] = pr;
        fprob[(size_t)k * D + d] = pr;
        psum += pr;
        if (d == 0) store_total_cost(p, q, k, s, D);
    }
    psum = block_reduce<0>(psum, scratch);
    if (tid == 0) p.wpart[((size_t)q * D + d) * p.wblocks_cap + blockIdx.x] = psum;
    tls.end();
}

// =====================================================================================================
// K8: PolicyImprovement::computeParameterUpdates (PolicyImprovement.cpp:584-711): probability-weighted
// noise sums sum_k P[k,d] * noise[k,d,t], the noise-adaptation numerator sum_k Pfull[k,d] * (n^T R n)[k,d]
// (quadratic forms from control_rows_kernel) and its denominator sum_k Pfull[k,d].  grid (chunks, D, Q); the
// CTA first normalises the weights of its chunk (the tables keep the unnormalised weights; read-backs divide), then
// thread t streams the chunk's noise rows with four independent accumulators.
// partial [Q][chunks][D][T+2]: update row, numerator, denominator.
// =====================================================================================================
constexpr int kUpdateThreads = 256;

// where apply_update_body finds the column sums [T + 2] (update row, adaptation numerator, sum of the weights)
enum UpdateSums : int {
    kSumsReduced = 0,            // updbuf: already summed (all-reduced over ranks, or per time step), normalised weights
    kSumsPartials = 1,           // the chunk partials of normalised weights (weighted_update_kernel)
    kSumsPartialsUnnormalised,   // the chunk partials of unnormalised weights (weights_update_kernel)
    kSumsRanksUnnormalised,      // s_cols already holds the unnormalised sums over all ranks (weights_update_peer_kernel)
};
__device__ __forceinline__ void apply_update_body(const LoopParams& p, int q, int d, UpdateSums sums, int nchunks, double* s_cols);

// column t of the chunk partials of (joint d, query q), added in chunk order: the result does not depend on which CTA
// finished last.  __ldcg: the partials may have been written by other CTAs of the running launch.  kUnroll: loads in flight
// per thread (16 where a single CTA sums all T + 2 columns, on the critical path of the update kernels).
template <int kUnroll>
__device__ __forceinline__ double chunk_column_sum(const LoopParams& p, int q, int d, int T, int D, int t, int nchunks)
{
    const double* col = p.partial + ((size_t)q * p.nchunks * D + d) * (T + 2) + t;
    const size_t stride = (size_t)D * (T + 2);
    double u = 0.0;
#pragma unroll kUnroll
    for (int c = 0; c < nchunks; ++c) u += __ldcg(col + (size_t)c * stride);
    return u;
}

// The chunk stream: 256 threads = two halves of 128, thread (half, lt) streams time step lt of every second row of the
// chunk (rows k_begin .. k_begin + nk) with 16 loads in flight, four accumulators; the halves are added in a fixed order.
// sp / sq: the chunk's row weights and weight * quad in shared memory.  Leaves out[0..T+1] = update row, adaptation
// numerator, sum of the weights (wsum_part: this thread's share).  T, D, sp and sq are the caller's: read again from p
// after the caller's stores, they would be loads of their own and change the update kernels' code.
// rollout_rows (the one-launch update kernels): when LoopParams::noise_from_rollouts is set, the rows are rollouts and
// noise_ = parameters_noise_ - parameters_ (PolicyImprovement.cpp:803-810) is formed here from the rollout row and theta —
// the same subtraction of the same two doubles the sampler would do.  theta is only written by the last chunk CTA of the
// launch, after every chunk CTA has finished streaming.  Otherwise the subtraction is of +0.0, the identity, which the
// compiler drops.
__device__ __forceinline__ void stream_chunk(const LoopParams& p, int q, int d, int T, int D, int k_begin, int nk, bool rollout_rows,
                                             const double* sp, const double* sq, double wsum_part, double* out, double* scratch,
                                             double* s_half)
{
    const int tid = threadIdx.x;
    const int half = tid >> 7, lt = tid & 127;
    for (int t0 = 0; t0 < T; t0 += 128) {
        const int t = t0 + lt;
        double acc = 0.0;
        if (t < T) {
            const bool from_rollouts = rollout_rows && p.noise_from_rollouts != 0;
            const double* nz = (from_rollouts ? p.rollouts : p.noise) + (((size_t)q * p.slots + k_begin) * D + d) * T + t;
            const double th_t = from_rollouts ? p.theta_all[((size_t)q * D + d) * p.N + kPad + t] : 0.0;
            const size_t stride = (size_t)D * T;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
            int k = half;
            for (; k + 30 < nk; k += 32) {       // rows k, k+2, ..., k+30
                double v[16];
#pragma unroll
                for (int u = 0; u < 16; ++u) v[u] = nz[(size_t)(k + 2 * u) * stride] - th_t;
#pragma unroll
                for (int u = 0; u < 16; u += 4) {
                    a0 += v[u] * sp[k + 2 * u]; a1 += v[u + 1] * sp[k + 2 * u + 2];
                    a2 += v[u + 2] * sp[k + 2 * u + 4]; a3 += v[u + 3] * sp[k + 2 * u + 6];
                }
            }
            for (; k < nk; k += 2) a0 += (nz[(size_t)k * stride] - th_t) * sp[k];
            acc = (a0 + a1) + (a2 + a3);
        }
        if (half != 0) s_half[lt] = acc;       // the second half (half is 0 or 1 with 256 threads)
        __syncthreads();
        if (half == 0 && t < T) out[t] = acc + s_half[lt];
        __syncthreads();
    }
    double numer = 0.0;
    for (int k = tid; k < nk; k += blockDim.x) numer += sq[k];
    numer = block_reduce<0>(numer, scratch);
    wsum_part = block_reduce<0>(wsum_part, scratch);
    if (tid == 0) { out[T] = numer; out[T + 1] = wsum_part; }
}

// chunk CTAs per (joint, query): gridDim.x of a (chunks, D, Q) grid, p.nchunks for weights_update_peer_kernel's
// one-dimensional grid.  Read where it is used: held from before the __threadfence below, it costs a register.
template <bool kPeer>
__device__ __forceinline__ unsigned int chunk_ctas(const LoopParams& p)
{
    return kPeer ? (unsigned int)p.nchunks : gridDim.x;
}

// The LAST chunk CTA of a (joint, query) to finish — found with a ticket counter after a __threadfence — runs apply(),
// when every chunk's partials are visible, and resets the ticket for the next launch.  D is the caller's copy of p.D and
// s_last the caller's __shared__ int: declared here, it would reorder the caller's shared memory and change its code.
template <bool kPeer, class Apply>
__device__ __forceinline__ void last_chunk_cta(const LoopParams& p, int q, int d, int D, int& s_last, Apply apply)
{
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.done_counter + (size_t)q * D + d, 1u) == chunk_ctas<kPeer>(p) - 1u) ? 1 : 0;
    __syncthreads();
    if (s_last) {
        __threadfence();
        apply();
        if (threadIdx.x == 0) p.done_counter[(size_t)q * D + d] = 0u;
    }
}

// fuse_apply (single GPU): the last chunk CTA also does the work of apply_update_kernel.  One launch and one drain / fill
// gap less per iteration.
// dynamic shared memory: max(2 * chunk, T + 2 + N) doubles (the last CTA of a joint also stages the updated row: apply_update_body).
__global__ void __launch_bounds__(kUpdateThreads)
weighted_update_kernel(const __grid_constant__ LoopParams p, int fuse_apply)
{
    extern __shared__ double smem[];   // [chunk] probabilities, [chunk] fprob * quad ; later [T + 2] column sums
    __shared__ double scratch[32];
    __shared__ double s_half[128];
    __shared__ int s_last;
    const int d = blockIdx.y, q = blockIdx.z, c = blockIdx.x;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 3);
    const int T = p.T, D = p.D, tid = threadIdx.x;
    const int k_begin = c * p.chunk, k_end = min(p.num_local, (c + 1) * p.chunk);
    const int nk = k_end - k_begin;
    double* sp = smem;
    double* sq = smem + p.chunk;
    if (tid < 32) {     // sum of the weights of joint d, partials in block order within a fixed butterfly
        const double* part = p.wpart + ((size_t)q * D + d) * p.wblocks_cap;
        double v = 0.0;
        for (int b = tid; b < p.wblocks; b += 32) v += part[b];
        v = warp_sum(v);
        if (tid == 0) scratch[0] = v;
    }
    __syncthreads();
    const double psum = scratch[0];
    __syncthreads();
    double fsum_part = 0.0;
    for (int k = k_begin + tid; k < k_end; k += blockDim.x) {
        const int g = (k == p.noiseless_slot) ? p.noiseless_gslot : ((k < p.num_gen) ? p.gen_offset + k : k);
        const size_t o = ((size_t)q * p.gslots + g) * D + d;
        const double pr = p.prob[o] / psum;       // probabilities_[d] = p / p_sum  (:546-549); full_probabilities_ alike (:575-578)
        // the noise-less rollout is replicated on every rank: only the first rank counts it in the denominator
        if (!(k == p.noiseless_slot && p.gen_offset != 0)) fsum_part += pr;
        double w = pr, fq = 0.0;
        if (k == p.noiseless_slot) w = 0.0;       // zero noise: contributes nothing (PolicyImprovement.cpp:407-410)
        else if (p.use_noise_adaptation) fq = pr * p.sums[((size_t)q * p.gslots + g) * p.sumw + 1 + 2 * D + d];
        sp[k - k_begin] = w;
        sq[k - k_begin] = fq;
    }
    __syncthreads();
    double* out = p.partial + (((size_t)q * p.nchunks + c) * D + d) * (T + 2);
    stream_chunk(p, q, d, T, D, k_begin, nk, false, sp, sq, fsum_part, out, scratch, s_half);
    if (fuse_apply)
        last_chunk_cta<false>(p, q, d, D, s_last, [&] { apply_update_body(p, q, d, kSumsPartials, (int)gridDim.x, smem); });
    tls.end();
}

// =====================================================================================================
// Rollout sharding without a collective library on the data path (SURVEY.md 8e, DESIGN.md 8).  Every rank maps the
// other ranks' MAILBOX (cudaIpc, engine.cu: setup_peer_exchange) and the two exchanges of an iteration happen inside ONE
// kernel, weights_update_peer_kernel, as plain stores over NVLink and spins on the rank's own memory:
//   A. the min / max of cumulative_costs_[d] over the rank's own rollouts (2 doubles per joint) -> every rank takes the
//      min / max over the ranks: the same two numbers the single-GPU scan finds, so the weights are bit-identical;
//   B. the rank's unnormalised partial sums [T + 2] per joint (update row, adaptation numerator, sum of the weights) ->
//      every rank adds the rows in RANK ORDER (deterministic, identical on all ranks) and applies the update.
// Transport: every double travels as two self-validating 8-byte words {epoch : 32 | half of the bits : 32} (the "LL"
// scheme: an aligned 8-byte store is atomic, so a word whose tag equals the exchange's epoch IS the data).  No fence, no
// separate flag, no release / acquire pair: one NVLink crossing per exchange.  (The first version — data, then
// __threadfence_system, then a release flag — cost 13 us per iteration on two B200s: MEMBAR.SYS is slow.)  The epoch is
// one per iteration, the same on every rank; slots are double buffered by its parity (a rank reaches exchange A of epoch
// e + 2 only after every rank has published B of e + 1, i.e. after it finished reading epoch e).  A spin that lasts 4 s
// sets the error flag, which every later wait honours: a missing rank costs seconds, never a hung GPU.
// Mailbox layout (bytes from the base; W ranks, D joints, T time steps):
//   A [2][W][D][2 doubles as 4 words] | B [2][W][D][T + 2 doubles as 2 (T + 2) words] | barrier [W] u32
// =====================================================================================================
constexpr int kMaxPeers = 8;
struct PeerExchange {
    unsigned char* box[kMaxPeers];   // mailbox of every rank, own included (own: plain device memory)
    int32_t world, rank;
    uint32_t epoch;                  // this iteration's exchange number (>= 1) unless epoch_ptr is set
    const uint32_t* epoch_ptr;       // device-side epoch (iterations replayed from a CUDA graph), or null
    int32_t* error;                  // device flag: a wait timed out
    int32_t D, T;
};
__host__ __device__ inline size_t peer_off_b(int W, int D) { return (size_t)2 * W * D * 32; }
__host__ __device__ inline size_t peer_off_barrier(int W, int D, int T) { return peer_off_b(W, D) + (size_t)2 * W * D * (T + 2) * 16; }
__host__ __device__ inline size_t peer_box_bytes(int W, int D, int T) { return peer_off_barrier(W, D, T) + 64; }

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// waits until *flag has reached `epoch`; false (and the error flag) after 4 s, or at once when the flag is already set
__device__ __forceinline__ bool peer_wait(const uint32_t* flag, uint32_t epoch, int32_t* error)
{
    unsigned long long t0 = 0;
    int polls = 0;
    while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
        if (++polls == 256) {
            polls = 0;
            if (*(volatile int32_t*)error) return false;
            const unsigned long long now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) { atomicExch(error, 1); return false; }
        }
    }
    return true;
}
// one double as two tagged words, 16 bytes at dst (16-byte aligned)
__device__ __forceinline__ void ll_store(unsigned char* dst, double v, uint32_t epoch)
{
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v), tag = (unsigned long long)epoch << 32;
    const unsigned long long w0 = tag | (bits & 0xffffffffull), w1 = tag | (bits >> 32);
    asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(dst), "l"(w0), "l"(w1) : "memory");
}
// spins until both words at src carry `epoch`; 0.0 (and the error flag) after 4 s
__device__ __forceinline__ double ll_load(const unsigned char* src, uint32_t epoch, int32_t* error)
{
    unsigned long long w0, w1, t0 = 0;
    int polls = 0;
    for (;;) {
        asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(src) : "memory");
        if ((uint32_t)(w0 >> 32) == epoch && (uint32_t)(w1 >> 32) == epoch) break;
        if (++polls == 256) {
            polls = 0;
            if (*(volatile int32_t*)error) return 0.0;
            const unsigned long long now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ull) { atomicExch(error, 1); return 0.0; }
        }
    }
    return __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
}

// all ranks meet on the device (timer brackets of a sharded run start together); one warp
__global__ void peer_barrier_kernel(const __grid_constant__ PeerExchange px, uint32_t ticket)
{
    const int r = threadIdx.x;
    if (r >= px.world) return;
    const size_t off = peer_off_barrier(px.world, px.D, px.T);
    st_release_sys(reinterpret_cast<uint32_t*>(px.box[r] + off) + px.rank, ticket);
    peer_wait(reinterpret_cast<const uint32_t*>(px.box[px.rank] + off) + r, ticket, px.error);
}

// K7 + K8 + K9 in one launch: computeRolloutProbabilities, computeParameterUpdates and updateParameters.  256 threads
// per CTA, one CTA per (chunk, joint, query).  Every CTA finds the min / max of its joint's costs itself — a coalesced
// scan of the compact mirrors s_compact / c_compact (2 x 8 K' bytes, L2 hits after the first CTA) — weighs the rollouts
// of its chunk (exp), streams their noise rows, and leaves the UNNORMALISED partial sums
//   out[t] = sum_k p_k noise_k[t],  out[T] = sum_k p_k (n^T R n)_k,  out[T+1] = sum_k p_k
// in `partial`; the last CTA of the (joint, query) adds the chunks in chunk order and divides by sum_k p_k
// (probabilities_ = p / p_sum, PolicyImprovement.cpp:546-549; the division commutes with the sum over k up to
// rounding).  Replaces rollout_weights_kernel -> gap -> weighted_update_kernel: one launch, one exposed L2 scan less.
// kPeer (rollout sharding, px): the scan covers this rank's rollouts and the noise-less one, exchange A makes the min /
// max global; exchange B adds the ranks' sums in rank order in front of the apply.
// dynamic shared memory: max(2 * chunk, T + 2 + N) doubles.
template <bool kPeer>
__device__ __forceinline__ void weights_update_body(const LoopParams& p, const PeerExchange* px, int c, int d, int q)
{
    extern __shared__ double smem[];   // [chunk] weights, [chunk] weight * quad ; later [T + 2] column sums
    __shared__ double scratch[32];
    __shared__ double s_half[128];
    __shared__ int s_last;
    pdl_trigger_and_wait();
    if (p.counters && c == 0 && d == 0 && q == 0 && threadIdx.x == 0) p.counters[0] += 1u;   // next iteration number (graph replay)
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 3);
    const int T = p.T, D = p.D, tid = threadIdx.x, n = p.num_rollouts;
    const int k_begin = c * p.chunk, k_end = min(p.num_local, (c + 1) * p.chunk);
    const int nk = k_end - k_begin;
    double* sp = smem;
    double* sq = smem + p.chunk;
    uint32_t epoch = 0;
    if constexpr (kPeer) epoch = px->epoch_ptr ? __ldcg(px->epoch_ptr) : px->epoch;
    const int parity = (int)(epoch & 1u);
    if (c == 0 && d == 0 && p.noiseless_slot >= 0) materialise_noiseless(p, q, tid, blockDim.x);

    // ---- min / max of cumulative_costs_[d] = S + C_d over all rollouts (PolicyImprovement.cpp:501-513) ----
    const double* S = p.s_compact + (size_t)q * p.gslots;
    const double* C = p.c_compact + ((size_t)q * D + d) * p.gslots;
    const double* nl = p.nl_sums + (size_t)q * p.sumw;
    auto cum_of = [&](int g) { return (g == p.noiseless_gslot) ? 1.0 * (nl[0] + nl[1 + d]) : 1.0 * (S[g] + C[g]); };
    double mn = 1e300, mx = -1e300;
    if constexpr (kPeer) {     // this rank's rollouts and the noise-less one
#pragma unroll 8
        for (int k = tid; k < p.num_gen; k += kUpdateThreads) {
            const double cum = cum_of(p.gen_offset + k);
            mn = fmin(mn, cum); mx = fmax(mx, cum);
        }
        if (tid == 0 && p.noiseless_gslot >= 0) { const double cum = cum_of(p.noiseless_gslot); mn = fmin(mn, cum); mx = fmax(mx, cum); }
    } else {
#pragma unroll 8
        for (int k = tid; k < n; k += kUpdateThreads) {
            const double cum = cum_of(k);
            mn = fmin(mn, cum); mx = fmax(mx, cum);
        }
    }
    mn = block_reduce<1>(mn, scratch); mx = block_reduce<2>(mx, scratch);
    if constexpr (kPeer) {     // ---- exchange A: every rank takes the min / max over the ranks ----
        __shared__ double s_mm[2 * kMaxPeers];
        const int W = px->world, rank = px->rank;
        if (c == 0 && tid < W && tid != rank) {
            unsigned char* dst = px->box[tid] + (((size_t)parity * W + rank) * D + d) * 32;
            ll_store(dst, mn, epoch);
            ll_store(dst + 16, mx, epoch);
        }
        if (tid < W) {
            double vmn = mn, vmx = mx;
            if (tid != rank) {
                const unsigned char* src = px->box[rank] + (((size_t)parity * W + tid) * D + d) * 32;
                vmn = ll_load(src, epoch, px->error);
                vmx = ll_load(src + 16, epoch, px->error);
            }
            s_mm[2 * tid] = vmn; s_mm[2 * tid + 1] = vmx;
        }
        __syncthreads();
        for (int r = 0; r < W; ++r) { mn = fmin(mn, s_mm[2 * r]); mx = fmax(mx, s_mm[2 * r + 1]); }
    }
    double den = mx - mn;
    if (den < 1e-8) den = 1e-8;
    const double h = p.cost_scaling_h;

    // ---- unnormalised weights of this chunk ----
    double psum_part = 0.0;
    for (int k = k_begin + tid; k < k_end; k += blockDim.x) {
        // a rank of a sharded engine reuses no rollouts: every slot but the noise-less one is a generated rollout
        const int g = (k == p.noiseless_slot) ? p.noiseless_gslot : ((kPeer || k < p.num_gen) ? p.gen_offset + k : k);
        const double pr = 1.0 * exp(((-h) * (cum_of(g) - mn)) / den);      // importance_weight_ = 1
        const size_t o = ((size_t)q * p.gslots + g) * D + d;
        p.prob[o] = pr;
        p.fprob[o] = pr;
        // the noise-less rollout is replicated on every rank: only the first rank counts it in the sum of the weights
        if (!(kPeer && k == p.noiseless_slot && px->rank != 0)) psum_part += pr;
        double w = pr, fq = 0.0;
        if (k == p.noiseless_slot) w = 0.0;       // zero noise: contributes nothing (PolicyImprovement.cpp:407-410)
        else if (p.use_noise_adaptation) fq = pr * p.sums[((size_t)q * p.gslots + g) * p.sumw + 1 + 2 * D + d];
        sp[k - k_begin] = w;
        sq[k - k_begin] = fq;
        if (d == 0) store_total_cost(p, q, g, cost_row(p, q, g), D);
    }
    __syncthreads();
    double* out = p.partial + (((size_t)q * p.nchunks + c) * D + d) * (T + 2);
    stream_chunk(p, q, d, T, D, k_begin, nk, true, sp, sq, psum_part, out, scratch, s_half);

    last_chunk_cta<kPeer>(p, q, d, D, s_last, [&] {
        if constexpr (kPeer) {
            // ---- exchange B: this rank's sums in chunk order -> every mailbox; then all ranks' rows in rank order ----
            const int W = px->world, rank = px->rank;
            const size_t offb = peer_off_b(W, D);
            for (int t = tid; t < T + 2; t += blockDim.x) {
                const double mine = chunk_column_sum<8>(p, q, d, T, D, t, (int)chunk_ctas<kPeer>(p));
                for (int r = 0; r < W; ++r)
                    if (r != rank) ll_store(px->box[r] + offb + ((((size_t)parity * W + rank) * D + d) * (T + 2) + t) * 16, mine, epoch);
                double u = 0.0;
                for (int r = 0; r < W; ++r)
                    u += (r == rank) ? mine : ll_load(px->box[rank] + offb + ((((size_t)parity * W + r) * D + d) * (T + 2) + t) * 16, epoch, px->error);
                smem[t] = u;
            }
            apply_update_body(p, q, d, kSumsRanksUnnormalised, (int)chunk_ctas<kPeer>(p), smem);
        } else {
            apply_update_body(p, q, d, kSumsPartialsUnnormalised, (int)chunk_ctas<kPeer>(p), smem);
        }
    });
    tls.end();
}

// single GPU, no rollout reuse: grid (chunks, D, Q)
__global__ void __launch_bounds__(kUpdateThreads)
weights_update_kernel(const __grid_constant__ LoopParams p)
{
    const int d = blockIdx.y, q = blockIdx.z, c = blockIdx.x;
    weights_update_body<false>(p, nullptr, c, d, q);
}

// a rollout-sharded engine (one query): grid nchunks * D CTAs in one dimension.  The D CTAs that publish exchange A come
// first in dispatch order and no CTA ever waits for another CTA of its own grid before publishing, so the spins cannot
// starve a publisher of an SM.
__global__ void __launch_bounds__(kUpdateThreads)
weights_update_peer_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ PeerExchange px)
{
    const int D = p.D, nchunks = p.nchunks;
    int c, d;
    if ((int)blockIdx.x < D) { c = 0; d = blockIdx.x; }
    else { const int r = blockIdx.x - D; d = r / (nchunks - 1); c = 1 + (r - d * (nchunks - 1)); }
    weights_update_body<true>(p, &px, c, d, 0);
}

// -----------------------------------------------------------------------------------------------------
// Per-time-step costs: Stomp::setCostCumulation(false).  cumulative_costs_[d] = total_costs_[d] = state + control_d per
// time step (PolicyImprovement.cpp:473-481); min / max per joint over all rollouts AND time steps (:501-513);
// probabilities per time step, normalised over the rollouts of that time step (:530-549); the update row is
// sum_r noise[r][d][t] * P[r][d][t] (:590-596).  full_probabilities_ (noise adaptation) stay those of the summed costs
// and come from rollout_weights_kernel.  Not a shipped configuration: simple kernels, rollouts walked in index order
// like the reference does.  Needs the per-time-step control costs (control_costs, folded) of every slot.
// -----------------------------------------------------------------------------------------------------
// cost-to-go per (rollout, joint): cum(T-1) = total(T-1), cum(t) = total(t) + cum(t+1); thread per (rollout, joint)
__global__ void __launch_bounds__(128)
pertimestep_suffix_kernel(const __grid_constant__ LoopParams p)      // grid (ceil(n D / 128), Q)
{
    const int q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D, n = p.num_local;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * D) return;
    const int k = e / D, d = e - k * D;
    const double* st = p.state_costs + ((size_t)q * p.slots + k) * T;
    const double* cc = p.control_costs + (((size_t)q * p.slots + k) * D + d) * T;
    double* out = p.pt_cum + (((size_t)q * p.slots + k) * D + d) * T;
    double acc = 1.0 * (st[T - 1] + cc[T - 1]);
    out[T - 1] = acc;
    for (int t = T - 2; t >= 0; --t) {
        acc = 1.0 * (st[t] + cc[t]) + acc;
        out[t] = acc;
    }
}

__global__ void __launch_bounds__(1024)
pertimestep_minmax_kernel(const __grid_constant__ LoopParams p)      // grid (D, Q)
{
    __shared__ double scratch[32];
    const int d = blockIdx.x, q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D, n = p.num_local;
    double mn = 1e300, mx = -1e300;
    for (int e = threadIdx.x; e < n * T; e += blockDim.x) {
        const int k = e / T, t = e - k * T;
        const double c = p.forward_cumulation ? p.pt_cum[(((size_t)q * p.slots + k) * D + d) * T + t]
                                              : 1.0 * (p.state_costs[((size_t)q * p.slots + k) * T + t] + p.control_costs[(((size_t)q * p.slots + k) * D + d) * T + t]);
        mn = fmin(mn, c); mx = fmax(mx, c);
    }
    mn = block_reduce<1>(mn, scratch); mx = block_reduce<2>(mx, scratch);
    if (threadIdx.x == 0) {
        double den = mx - mn;
        if (den < 1e-8) den = 1e-8;
        p.pt_minden[((size_t)q * D + d) * 2] = mn;
        p.pt_minden[((size_t)q * D + d) * 2 + 1] = den;
    }
}

__global__ void __launch_bounds__(128)
pertimestep_update_kernel(const __grid_constant__ LoopParams p)      // grid (ceil(T / 128), D, Q)
{
    const int d = blockIdx.y, q = blockIdx.z;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D, n = p.num_local;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    double mn = p.pt_minden[((size_t)q * D + d) * 2], den = p.pt_minden[((size_t)q * D + d) * 2 + 1];
    const double h = p.cost_scaling_h;
    double* upd = p.updbuf + ((size_t)q * D + d) * (T + 2);
    if (t < T) {
        auto cost_of = [&](int k) {
            if (p.forward_cumulation) return p.pt_cum[(((size_t)q * p.slots + k) * D + d) * T + t];
            return 1.0 * (p.state_costs[((size_t)q * p.slots + k) * T + t] + p.control_costs[(((size_t)q * p.slots + k) * D + d) * T + t]);
        };
        if (p.per_timestep_minmax) {     // min / max over the rollouts of THIS time step (the variant at PolicyImprovement.cpp:518-528)
            double lo = cost_of(0), hi = lo;
            for (int k = 1; k < n; ++k) { const double c = cost_of(k); lo = fmin(lo, c); hi = fmax(hi, c); }
            mn = lo;
            den = hi - lo;
            if (den < 1e-8) den = 1e-8;
        }
        // the unnormalised weights are parked in pt_prob (one exp per rollout), normalised in the second walk
        double* pt = p.pt_prob + (((size_t)q * p.gslots) * D + d) * T + t;
        const size_t pt_stride = (size_t)D * T;
        double psum = 0.0;
        for (int k = 0; k < n; ++k) {
            const double w = 1.0 * exp(((-h) * (cost_of(k) - mn)) / den);      // importance_weight_ = 1
            pt[(size_t)k * pt_stride] = w;
            psum += w;
        }
        double u = 0.0;
        for (int k = 0; k < n; ++k) {
            const double pr = pt[(size_t)k * pt_stride] / psum;
            pt[(size_t)k * pt_stride] = pr;
            u += p.noise[(((size_t)q * p.slots + k) * D + d) * T + t] * pr;     // the noise-less slot carries zero noise
        }
        upd[t] = u;
    }
    if (blockIdx.x == 0 && threadIdx.x < 32) {      // noise adaptation: sum_r Pfull (n^T R n), sum_r Pfull (:656-663)
        const double* part = p.wpart + ((size_t)q * D + d) * p.wblocks_cap;
        double wsum = 0.0;
        for (int b = 0; b < p.wblocks; ++b) wsum += part[b];
        double numer = 0.0, denom = 0.0;
        for (int k = threadIdx.x; k < n; k += 32) {
            const double pf = p.fprob[((size_t)q * p.gslots + k) * D + d] / wsum;
            denom += pf;
            if (k != p.noiseless_slot && p.use_noise_adaptation) numer += pf * p.sums[((size_t)q * p.gslots + k) * p.sumw + 1 + 2 * D + d];
        }
        numer = warp_sum(numer); denom = warp_sum(denom);
        if (threadIdx.x == 0) { upd[T] = numer; upd[T + 1] = denom; }
    }
}

// sum of the chunk partials in chunk order -> updbuf [Q][D][T+1]; only needed in front of the all-reduce
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const __grid_constant__ LoopParams p, int nchunks)
{
    const int d = blockIdx.x, q = blockIdx.y;
    if (query_frozen(p, q)) return;
    const int T = p.T, D = p.D;
    for (int t = threadIdx.x; t < T + 2; t += blockDim.x) p.updbuf[((size_t)q * D + d) * (T + 2) + t] = chunk_column_sum<8>(p, q, d, T, D, t, nchunks);
}

// =====================================================================================================
// K8 tail + K9: noise adaptation (PolicyImprovement.cpp:656-679) and CovariantMovementPrimitive::
// updateParameters (stomp/src/CovariantMovementPrimitive.cpp:476-479).  grid (D, Q).  sums: where the column sums
// come from (UpdateSums).
// =====================================================================================================
// s_cols: T + 2 doubles of shared memory.  Column sums first (all threads, 16 loads in flight each), then the update.
__device__ __forceinline__ void apply_update_body(const LoopParams& p, int q, int d, UpdateSums sums, int nchunks, double* s_cols)
{
    const int T = p.T, D = p.D, N = p.N;
    __syncthreads();
    if (p.nl_sums_next)       // the padding (start / goal) of the row whose control costs are taken at the end: requested now, off the critical path
        for (int i = threadIdx.x; i < 2 * kPad; i += blockDim.x) {
            const int j = i < kPad ? i : T + i;
            s_cols[(T + 2) + j] = p.theta_all[((size_t)q * D + d) * N + j];
        }
    if (sums != kSumsRanksUnnormalised)
        for (int t = threadIdx.x; t < T + 2; t += blockDim.x)
            s_cols[t] = (sums == kSumsReduced) ? p.updbuf[((size_t)q * D + d) * (T + 2) + t] : chunk_column_sum<16>(p, q, d, T, D, t, nchunks);
    __syncthreads();
    // unnormalised weights (weights_update_kernel, weights_update_peer_kernel): divide by their total, which is also what
    // the read-backs of the probabilities divide by
    const bool unnormalised = sums == kSumsPartialsUnnormalised || sums == kSumsRanksUnnormalised;
    const double psum = unnormalised ? s_cols[T + 1] : 1.0;
    if (unnormalised && threadIdx.x == 0) p.wpart[((size_t)q * D + d) * p.wblocks_cap] = psum;
    if (p.Mproj) {
        // parameter_updates_.row(0) = projection_matrix_ * row(0) (PolicyImprovement.cpp:706): normalise the row in
        // place first (the branch below then sees the finished row), every thread then forms its own dot product
        __syncthreads();
        for (int t = threadIdx.x; t < T; t += blockDim.x) {
            double u = s_cols[t];
            if (unnormalised) u = u / psum;
            u *= 1.0;
            u /= 1.0;
            s_cols[t] = u;
        }
        __syncthreads();
    }
    for (int t = threadIdx.x; t < T + 1; t += blockDim.x) {
        double u = s_cols[t];
        if (unnormalised && !(p.Mproj && t < T)) u = u / psum;
        if (t < T) {
            if (p.Mproj) {
                const double* mrow = p.Mproj + (size_t)t * T;
                double acc = 0.0;
                for (int j = 0; j < T; ++j) acc += mrow[j] * s_cols[j];
                u = acc;
            } else {
                // time-step weights and divisor are exactly 1 (PolicyImprovement.cpp:533,684-704)
                u *= 1.0;
                u /= 1.0;
            }
            p.updates[((size_t)q * D + d) * T + t] = u;
            double* th = p.theta_all + ((size_t)q * D + d) * N + kPad + t;
            const double updated = *th + 1.0 * u;
            *th = updated;
            if (p.nl_sums_next) s_cols[(T + 2) + kPad + t] = updated;       // the updated row, staged for its control costs below
        } else if (p.use_noise_adaptation) {
            const double denom = unnormalised ? s_cols[T + 1] / psum : s_cols[T + 1];
            p.fprob_sum[(size_t)q * D + d] = denom;
            const double frob_stddev = sqrt(u / (denom * T));
            const double update_rate = 0.2;
            double sd = (1.0 - update_rate) * p.sigma[(size_t)q * D + d] + update_rate * frob_stddev;
            if (sd < p.min_stddev[d]) sd = p.min_stddev[d];
            p.sigma[(size_t)q * D + d] = sd;
            store_sampler_coefficients(p, q, d, sd);
        }
    }
    // ---- control costs of the UPDATED row: the control half of the noise-less rollout (Stomp::doNoiselessRollout,
    // Stomp.cpp:253-272; noise = 0) is known the moment the parameters are — computed here, by the CTA that just wrote the
    // row, into the record the NEXT iteration reads; the state half rides on the next state kernel launch ----
    if (p.nl_sums_next) {
        double* s_row = s_cols + (T + 2);
        __syncthreads();
        if (threadIdx.x < 32) {
            const int lane = threadIdx.x;
            double C_d, cum_d;
            if (p.control_costs == nullptr && p.st_uniform) {
                // the shipped loop: interior rows from the staged row, the six padding-only rows from edge_cost (constants of
                // the solve, edge_rows_kernel) — no table walk on the critical path of the update kernel
                double c_sum = 0.0;
                for (int i = 3 + lane; i < N - 3; i += 32) c_sum += interior_row_cost<0, 6>(p, [&](int o) { return s_row[i - 3 + o]; });
                C_d = warp_sum(c_sum) + edge_cost_sum(p, q, d);
            } else {
                control_cost_sums(p, s_row, nullptr, lane, C_d, cum_d);
                control_cost_store(p, s_row, lane, p.nl_control + ((size_t)q * D + d) * T);
            }
            if (lane == 0) {
                double* nl = p.nl_sums_next + (size_t)q * p.sumw;
                nl[1 + d] = C_d; nl[1 + D + d] = C_d; nl[1 + 2 * D + d] = 0.0;
            }
        }
    }
}

// dynamic shared memory: T + 2 + N doubles
__global__ void __launch_bounds__(256)
apply_update_kernel(const __grid_constant__ LoopParams p, int sums, int nchunks)     // sums: UpdateSums
{
    extern __shared__ double smem[];
    const int d = blockIdx.x, q = blockIdx.y;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 4);
    apply_update_body(p, q, d, (UpdateSums)sums, nchunks, smem);
    tls.end();
}

// =====================================================================================================
// K10: Stomp::doNoiselessRollout (stomp/src/Stomp.cpp:253-272) + setNoiselessRolloutCosts
// (PolicyImprovement.cpp:401-419) and the wrapper's stop rule (src/wrappers/stomp/StompPlanner.cpp:107-118).
// One CTA per query; runs on the engine's side stream, overlapped with the next iteration's sampling and
// rollout costs (its result is first needed by the next rollout_weights_kernel).  The verdicts of the T states are
// the ones a state pass over the padded policy rows wrote to nl_state just before, on the same stream.
// =====================================================================================================
__global__ void __launch_bounds__(256)
noiseless_rollout_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ RobotParams robot,
                         const __grid_constant__ SdfParams sdf, const __grid_constant__ CostExtras extras)
{
    extern __shared__ double smem[];
    const int q = blockIdx.x;
    if (query_frozen(p, q)) return;
    TimelineScope tls(p, 5);
    const int T = p.T, D = p.D, N = p.N, tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    double* sx = smem;                      // [D][N]
    double* sstate = smem + (size_t)D * N;  // [T]
    double* ssum = sstate + T;              // [1 + 2D]
#pragma unroll 4
    for (int e = tid; e < D * N; e += blockDim.x) sx[e] = p.theta_all[(size_t)q * D * N + e];
    for (int t = tid; t < T; t += blockDim.x) sstate[t] = p.nl_state[(size_t)q * T + t];
    __syncthreads();
    if (extras.smooth || extras.joint_constraint) {     // alternative state costs of the noise-less states (see CostExtras)
        const SdfParams field = query_field(p.query_sdf, q, sdf);
        for (int t = tid; t < T; t += blockDim.x) {
            const double* xq = sx + kPad + t;
            sstate[t] = extra_state_cost(robot, field, extras, [&](int d) { return xq[(size_t)d * N]; }, sstate[t]);
            p.nl_state[(size_t)q * T + t] = sstate[t];
        }
        __syncthreads();
    }
    // control costs (noise = 0: parameters + 0.0 is exact) and sums
    for (int task = warp; task < D + 1; task += nwarps) {
        if (task < D) {
            double C_d, cum_d;
            control_cost_sums(p, sx + (size_t)task * N, sstate, lane, C_d, cum_d);
            control_cost_store(p, sx + (size_t)task * N, lane, p.nl_control + ((size_t)q * D + task) * T);
            if (lane == 0) { ssum[1 + task] = C_d; ssum[1 + D + task] = cum_d; ssum[1 + 2 * D + task] = 0.0; }
        } else {
            double s = 0.0;
            for (int t = lane; t < T; t += 32) s += sstate[t];
            s = warp_sum(s);
            if (lane == 0) ssum[0] = s;
        }
    }
    __syncthreads();
    for (int e = tid; e < p.sumw; e += blockDim.x) p.nl_sums_next[(size_t)q * p.sumw + e] = ssum[e];     // the record the next iteration reads
    if (tid == 0) {
        double cost = ssum[0];
        for (int d = 0; d < D; ++d) cost += ssum[1 + d];
        p.nl_total[q] = cost;
        if (cost < p.best_cost[q]) p.best_cost[q] = cost;
        const double improvement = cost - p.old_cost[q];
        p.old_cost[q] = cost;
        p.last_improvement[q] = improvement;
        const int recorded = p.iters_used[q] + 1;
        p.iters_used[q] = recorded;
        const bool stop_now = (cost < 1) && (fabs(improvement) < p.min_cost_improvement);
        if (stop_now) p.stop[q] = 1;
        if (p.note) {      // progress words in host memory (stomp_b200_solve paces its queue by them)
            volatile int* note = p.note + 2 * q;
            if (stop_now) note[1] = 1;
            note[0] = recorded;
        }
    }
    tls.end();
}

}  // namespace stomp_b200
