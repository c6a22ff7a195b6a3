// Host orchestration + C ABI (include/stomp_b200.h) of the B200 STOMP rollout loop.
//
// One engine = one GPU; a main stream plus two helper streams for the fallback paths (control-cost rows beside the state
// kernel; a two-kernel noise-less rollout under the next iteration's sampling).  The per-iteration sequence mirrors
// stomp::Stomp::runSingleIteration (reference src/planners/stomp/src/Stomp.cpp:274-301); shipped loop first, fallbacks after |:
//   doGenRollouts      -> [reuse_rollouts_kernel], then launch_generate_stage, in the shape generate_shape classifies the
//                         iteration into: sample_rollouts_banded_kernel (recurrence through the banded L^-1, control-cost rows
//                         fused; draws before it waits for the previous update kernel) | sample_rollouts_dmma_kernel (injected
//                         epsilon, factors without a band table) | shift_rollouts_kernel (injected unit noise)
//   doExecuteRollouts  -> a state pass (launch_state_pass, also for the noise-less rollout and stomp_b200_evaluate_states):
//                         stomp_b200_states_specialised (generated, state_codegen.hpp; static spheres once per scene by
//                         stomp_b200_static_spheres) | rollout_states_kernel; states_self_collision_kernel / the generated
//                         pair-rule kernel with a sphere-pair list; then state_cost_extras_kernel for the alternative costs
//   setRolloutCosts    -> inside the sampler | launch_generate_stage: control_rows_tile_kernel | control_rows_fast_kernel |
//                         control_rows_kernel, behind project_noise_dmma_kernel with use_projection; [reused_control_cost_kernel];
//                         all of them form rows, n^T R n terms and sums with the same functions (kernels.cuh: band_row_cost,
//                         interior_row_cost, quad_term, edge_cost_sum, store_row_sums)
//   improvePolicy + updateParameters
//                      -> launch_update_stage, in the shape update_shape classifies the iteration into: weights_update_kernel on
//                         one GPU, weights_update_peer_kernel (both exchanges over NVLink mailboxes) on rollout shards | with the
//                         NCCL exchange, rollout reuse or per-kernel profiling: [allgather] rollout_weights_kernel,
//                         weighted_update_kernel, [reduce_partials_kernel, allreduce], apply_update_kernel | per-time-step costs:
//                         rollout_weights_kernel, the pertimestep kernels, apply_update_kernel
//   doNoiselessRollout -> control costs in the update kernel's last CTA per joint, the T states as a tail of the next state kernel
//                         launch (alone at a join) | a state pass on the T states + noiseless_rollout_kernel (side stream)
// The rollout bookkeeping (PolicyImprovement.cpp:170-186,304-308) is host integer arithmetic and stays here.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <limits>
#include <set>
#include <string>
#include <vector>

#include <cuda_runtime.h>
#include <nccl.h>

#include "../../include/stomp_b200.h"
#include "../host/policy_core.hpp"
#include "kernels.cuh"
#include "sdf_builder.cuh"
#include "state_codegen.hpp"

using namespace stomp_b200;

namespace {

struct SigmaIt { double v[STOMP_B200_MAX_DIMS]; };

__global__ void set_sigma_by_value_kernel(const __grid_constant__ LoopParams p, const __grid_constant__ SigmaIt s)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= p.Q * p.D) return;
    if (query_frozen(p, e / p.D)) return;
    p.sigma[e] = s.v[e % p.D];
    store_sampler_coefficients(p, e / p.D, e % p.D, s.v[e % p.D]);
}

__global__ void reset_solve_state_kernel(const __grid_constant__ LoopParams p)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= p.Q) return;
    p.old_cost[q] = 0.0;
    p.last_improvement[q] = 0.0;
    p.best_cost[q] = 1.7976931348623157e308;
    p.stop[q] = 0;
    p.iters_used[q] = 0;
    p.nl_total[q] = 0.0;
    p.nl_valid[q] = 0;
}

// NCCL is bound at run time (dlopen) so that a single-GPU process never needs the library and a Python
// host that already loaded its own libnccl.so.2 shares it.
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool load(std::string& err)
    {
        if (lib) return true;
        lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) { err = std::string("dlopen(libnccl.so.2): ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllGather || !AllReduce || !GetErrorString) {
            err = "libnccl.so.2 lacks a required symbol";
            return false;
        }
        return true;
    }
};
NcclApi g_nccl;

struct ProfiledLaunch { int kernel; cudaEvent_t a, b; };

// STOMP_B200_SAMPLER at creation: "dmma" the contraction for on-device noise too, "banded" the recurrence for injected
// epsilon too; unset or any other value the default (generate_shape)
enum class SamplerSwitch { kDefault, kContraction, kRecurrence };

}  // namespace

struct stomp_b200_engine {
    stomp_b200_config cfg;
    int T = 0, D = 0, N = 0, Q = 0, slots = 0, gslots = 0, sumw = 0;
    int query_offset = 0;
    bool reuse_possible = false;
    cudaStream_t stream = nullptr;
    std::string last_error;
    std::vector<void*> allocations;
    std::set<const void*> smem_opted_in;   // kernels whose dynamic shared-memory limit was raised on this engine's device

    RobotParams robot;
    JointLimits limits;             // robot.lower / upper, for the sampling kernels
    SdfParams sdf;
    float* d_sdf = nullptr;
    size_t sdf_count = 0;
    double sdf_origin[3] = {0, 0, 0}, sdf_voxel = 0;
    CostExtras extras;              // stomp_b200_set_cost_extras; all zero: the shipped 0 / 1 state cost
    bool extras_on = false;
    SelfPairs self_pairs = {nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0};   // stomp_b200_set_self_collision; n == 0: world collisions only
    std::vector<void*> self_pair_buffers;
    // the pair rule inside a run-time specialised kernel (state_codegen.hpp: SelfPairStructure): structure, FP32 thresholds
    // (lo[P], hi[P], block[B]: the SelfBands kernel parameter) and the kernel, resolved at the first launch after a change
    codegen::SelfPairStructure self_structure;
    std::vector<float> self_bands;
    const codegen::SpecialisedKernel* spec_self = nullptr;
    bool spec_self_resolved = false;
    std::string spec_self_note;
    bool have_chain = false, have_spheres = false, have_sdf = false, have_matrices = false;
    std::vector<uint8_t> have_policy;

    LoopParams base;                // pointers + constants; per-iteration fields filled in iterate
    double* proj2[2] = {nullptr, nullptr};
    double* d_Lband = nullptr;               // [T][8] rows of L^-1 for the recurrence sampler
    SamplerSwitch sampler_switch = SamplerSwitch::kDefault;
    double* d_Mproj = nullptr; double* d_Minv = nullptr;   // projection_matrix_ / its inverse (use_projection only)
    double* state2[2] = {nullptr, nullptr};
    uint8_t* verdict2[2] = {nullptr, nullptr};
    int32_t* d_order = nullptr;
    int max_chunks = 1;
    int num_sms = 148;
    cudaStream_t side_stream = nullptr;      // noise-less rollout, overlapped with the next iteration's sampling + costs
    cudaEvent_t ev_applied = nullptr, ev_noiseless = nullptr;
    cudaStream_t rows_stream = nullptr;      // control-cost rows, side by side with the state kernel
    cudaEvent_t ev_sampled = nullptr, ev_rows = nullptr;
    // With the run-time specialised state kernel the owed rollout needs no kernel of its own: its control costs are
    // computed by the update kernel's last CTA per joint (apply_update_body), its T states ride on the next state kernel
    // launch as a tail (kinematics.cuh: NoiselessTail), whose last thread does the bookkeeping and the stop rule.  The
    // record of the rollout is double buffered: the update of iteration i writes the one iteration i + 1 reads.
    double* nl_sums2[2] = {nullptr, nullptr};
    uint32_t* d_nl_counter = nullptr;        // [Q] packed hit / finished-state counters of the tail

    // The host state an iteration (iterate_body) reads and writes, statistics and configuration aside.  Whole, so that a
    // CUDA graph replay can set it as the captured iteration left it and an abandoned capture can put it back (iterate_async).
    struct LoopState {
        // PolicyImprovement bookkeeping (PolicyImprovement.cpp:170-186) and what read-backs need of the last iteration
        int num_rollouts = 0;                    // num_rollouts_ after the previous iteration (global)
        int last_gen = 0, last_local = 0, last_noiseless_slot = -1;
        int last_wblocks = 1;                    // partial sums of the weights left in wpart by the last iteration
        bool last_noise_from_rollouts = false;   // the last iteration did not write `noise` (read-backs say so)
        bool noiseless_valid = false, adapted_valid = false;
        // The noise-less rollout of iteration i is LAUNCHED at the start of iteration i + 1 (or by the first call that needs
        // its result), not at the end of i: on the device nothing changes — it still runs on the side stream under the next
        // sampling — but an iteration then has the fork / join shape [noise-less of i-1 || sample, cost of i] -> update of i
        // that a CUDA graph can hold.
        bool nl_deferred = false;
        LoopParams nl_lp;                        // parameters of the iteration whose noise-less rollout is owed
        int nl_parity = 0;                       // nl_sums2[nl_parity] is what the next iteration reads
        bool noiseless_pending = false;          // ev_noiseless recorded and not yet waited for by the main stream
        int cur = 0;                             // proj2 / state2 / verdict2[cur] hold the last iteration's rollouts (reuse)
        bool edge_dirty = true;                  // edge_cost has to be recomputed (the policy was uploaded since)
        bool tables_gathered = true;             // rollout-indexed tables complete on this rank (peer mode gathers them lazily for read-backs)
        uint32_t peer_epoch = 0;                 // epoch of the last exchange queued (PeerExchange::epoch, LoopParams::counters[1])
    };
    LoopState loop;
    // steady-state iterations replayed from CUDA graphs (iterate_async): one per (honour_stop, record parity)
    struct IterationGraph {
        cudaGraphExec_t exec = nullptr;
        unsigned long long config_epoch = 0;
        int64_t launches = 0;                            // kernel nodes (what a replay adds to launch_count)
        LoopState after;                                 // the loop state the captured iteration left
    };
    IterationGraph graphs[2][2];             // [honour_stop][record parity]
    unsigned long long config_epoch = 1;     // bumped by every setter whose values are baked into kernel parameters
    // STOMP_B200_PDL=<mask> at creation: bit 0 sampler, 1 state kernel, 2 weights / update kernel launched as programmatic
    // dependents of the kernel before them (0: ordinary launches); bit 3 the noise-less tail launched alone at a join (84.8 ->
    // 83.9 us per isolated C3 iteration, profiles/r4j_pdl_tail.txt).  Default 15, all four.  The state kernel's edge pays only
    // with its largest-L1 preference (resolve_state_kernel): without it its CTAs become resident beside the sampler's and run
    // their gathers against a sliver of L1 (16.5 -> 34 us, profiles/r3r_pdl_edges.txt); with it the sampler -> state gap goes
    // from 3.1 to 1.1 us and the kernel keeps its 16.9 us (isolated C3 iteration 71.8 -> 69.4 us, profiles/r6a_*).
    int pdl_mask = 15;
    bool graphs_allowed = true;              // STOMP_B200_GRAPH=0 at creation switches the replay off
    bool timer_armed = false, timer_end_recorded = false;   // stomp_b200_timer_begin .. _end: stomp_b200_run records the end event itself
    bool graph_over_overlap = false;         // STOMP_B200_GRAPH=2: replay graphs even where plain launches would overlap the sampler with the update kernel
    bool early_sampler = true;               // STOMP_B200_SAMPLER_EARLY=0: the sampler waits for its predecessor before it draws (kernels.cuh)
    int eligible_streak = 0;                 // graph-eligible iterations run un-captured since the configuration last changed
    unsigned long long streak_epoch = 0;
    uint32_t* d_counters = nullptr;          // [0] iteration, [1] exchange epoch (LoopParams::counters)
    long long dev_iteration_next = -1;       // value counters[0] will hold when the queued work has run; -1 unknown
    long long dev_epoch_next = -1;           // likewise counters[1] (the epoch of the LAST exchange queued)
    int64_t graph_launches = 0;
    double* d_theta_all_init = nullptr;   // policy as uploaded by set_policy (restored by begin_solve? no: the policy persists)

    bool solving = false;
    bool fuse_weights_allowed = true;   // STOMP_B200_FUSE_WEIGHTS=0 at creation keeps K7 / K8 / K9 as separate kernels
    // state kernel specialised to the robot structure (state_codegen.hpp); resolved at the first iteration after
    // the chain / spheres / SDF changed
    const codegen::SpecialisedKernel* spec = nullptr;
    bool spec_resolved = false;
    int32_t* d_static_hit = nullptr;         // verdict of the spheres no joint value moves (stomp_b200_static_spheres), rewritten whenever the state kernel is resolved
    std::string spec_note;          // why the generic kernel is in use, when it is

    // pinned host mirrors of the per-query scalars
    double* h_cost = nullptr; uint8_t* h_valid = nullptr; int32_t* h_stop = nullptr; int32_t* h_iters = nullptr;
    double* h_impr = nullptr;
    unsigned char* h_scalars = nullptr;      // the pinned block the five mirrors above point into
    unsigned char* d_scalars = nullptr;      // its device counterpart (LoopParams nl_total / last_improvement / stop / iters_used / nl_valid)
    size_t scalar_bytes = 0;
    // Progress words the device writes straight into host memory (mapped, pinned): [Q][2] = (noise-less rollouts recorded,
    // stopped).  stomp_b200_solve queues iterations against them — a bounded number ahead of the device — instead of
    // synchronising every poll_every iterations: no bubbles, at most `solve_ahead` no-op iterations behind the stop.
    volatile int32_t* h_note = nullptr;
    int solve_ahead = 1;                     // STOMP_B200_SOLVE_AHEAD at creation; 0: the synchronising poll loop
    // results of the last read-back, valid until something is queued again: finish_solve after solve touches no device
    bool scalars_fresh = false, solution_fresh = false;
    bool note_writers_in_flight = false;     // kernels queued since the last synchronisation of the main stream
    double* h_solution = nullptr;            // pinned [Q][D][T], allocated on first use
    // pinned staging of stomp_b200_set_policies: [Q][D*N] then [Q][D*T]; a slot is rewritten only after its copy has gone out
    double* h_policy = nullptr;
    std::vector<uint8_t> policy_in_flight;
    cudaEvent_t ev_policy = nullptr;

    // measurement
    bool profiling = false;
    std::vector<ProfiledLaunch> pending;
    double kernel_ms[STOMP_B200_KERNEL_COUNT] = {0};
    int64_t kernel_launches[STOMP_B200_KERNEL_COUNT] = {0};
    int64_t launch_count = 0;
    cudaEvent_t timer_a = nullptr, timer_b = nullptr;

    // in-pipeline timeline: ring of the last kTimelineRing iterations
    unsigned long long* d_timeline = nullptr;
    bool timeline_on = false;
    long long timeline_count = 0;

    ncclComm_t comm = nullptr;
    // rollout sharding over peer-mapped mailboxes (kernels.cuh: weights_update_peer_kernel); NCCL stays the bootstrap, the
    // read-back gather and the fallback (STOMP_B200_EXCHANGE=nccl, or cudaIpc unavailable)
    PeerExchange px;
    bool peer_ready = false;
    uint32_t barrier_ticket = 0;
    void* peer_box_own = nullptr;
    std::vector<void*> peer_opened;
    int32_t* d_peer_error = nullptr; int32_t* h_peer_error = nullptr;
    std::string exchange_note = "single GPU: no exchange";

    // grow-only scratch of stomp_b200_evaluate_states
    double* eval_theta = nullptr; double* eval_cost = nullptr; uint8_t* eval_verdict = nullptr; uint8_t* eval_valid = nullptr;
    size_t eval_cap_theta = 0, eval_cap_states = 0, eval_cap_traj = 0;
};
constexpr int kTimelineRing = 64;

namespace {

#define CUDA_TRY(e, call)                                                                                    \
    do {                                                                                                     \
        cudaError_t _err = (call);                                                                           \
        if (_err != cudaSuccess) {                                                                           \
            (e)->last_error = std::string(#call) + ": " + cudaGetErrorString(_err);                          \
            return _err == cudaErrorMemoryAllocation ? STOMP_B200_ERR_OUT_OF_MEMORY : STOMP_B200_ERR_CUDA;   \
        }                                                                                                    \
    } while (0)

#define NCCL_TRY(e, call)                                                                \
    do {                                                                                 \
        ncclResult_t _r = (call);                                                        \
        if (_r != ncclSuccess) {                                                         \
            (e)->last_error = std::string(#call) + ": " + g_nccl.GetErrorString(_r);     \
            return STOMP_B200_ERR_NCCL;                                                  \
        }                                                                                \
    } while (0)

int fail(stomp_b200_engine* e, int code, const char* msg)
{
    if (e) e->last_error = msg;
    return code;
}

template <class Tp>
int dev_alloc(stomp_b200_engine* e, Tp** out, size_t count)
{
    void* p = nullptr;
    CUDA_TRY(e, cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(Tp)));
    CUDA_TRY(e, cudaMemsetAsync(p, 0, std::max<size_t>(count, 1) * sizeof(Tp), e->stream));
    e->allocations.push_back(p);
    *out = static_cast<Tp*>(p);
    return 0;
}

struct Scope {   // brackets one kernel launch with events when profiling is on
    stomp_b200_engine* e; int kernel; cudaEvent_t a = nullptr, b = nullptr;
    Scope(stomp_b200_engine* e_, int k) : e(e_), kernel(k)
    {
        if (e->profiling) {
            cudaEventCreate(&a); cudaEventCreate(&b);
            cudaEventRecord(a, e->stream);
        }
    }
    ~Scope()
    {
        e->launch_count++;
        e->kernel_launches[kernel]++;
        if (e->profiling) {
            cudaEventRecord(b, e->stream);
            e->pending.push_back({kernel, a, b});
        }
    }
};

void resolve_profile(stomp_b200_engine* e)
{
    for (auto& pl : e->pending) {
        float ms = 0.f;
        cudaEventSynchronize(pl.b);
        if (cudaEventElapsedTime(&ms, pl.a, pl.b) == cudaSuccess) e->kernel_ms[pl.kernel] += ms;
        cudaEventDestroy(pl.a);
        cudaEventDestroy(pl.b);
    }
    e->pending.clear();
}

// launch with programmatic stream serialisation (the kernel contains griddepcontrol.wait: kernels.cuh, pdl_trigger_and_wait)
cudaError_t launch_dependent(const stomp_b200_engine* e, int which, const void* kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t stream, void** args)
{
    cudaLaunchConfig_t cfg;
    std::memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr;
    std::memset(&attr, 0, sizeof attr);
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    // A dependent's CTAs become resident wherever room is while the kernel before it drains.  A grid that fills the GPU
    // anyway loses nothing; a small one gets packed onto the few SMs that were free first and runs slower than the gap it
    // saved (sampler of a 2048-rollout shard: 12.8 -> 18.6 us, profiles/r3u_pdl_two_gpus.txt): those launch the ordinary way.
    const long long ctas = (long long)grid.x * grid.y * grid.z;
    const bool fills = which == 0 ? ctas >= 5LL * e->num_sms : (which == 2 ? ctas >= (long long)e->num_sms : true);
    cfg.numAttrs = (((e->pdl_mask >> which) & 1) && fills) ? 1 : 0;
    return cudaLaunchKernelExC(&cfg, kernel, args);
}

int check_launch(stomp_b200_engine* e, const char* what)
{
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        e->last_error = std::string(what) + ": " + cudaGetErrorString(err);
        return STOMP_B200_ERR_CUDA;
    }
    return 0;
}

codegen::StateKernelOptions state_kernel_options(const stomp_b200_engine* e);

// the specialised kernel with the pair rule for the pair list as it is now, or null (then states_self_collision_kernel runs)
void resolve_self_kernel(stomp_b200_engine* e)
{
    if (e->spec_self_resolved) return;
    e->spec_self_resolved = true;
    e->spec_self = nullptr;
    const char* mode = std::getenv("STOMP_B200_SELF");
    if (mode && std::strcmp(mode, "generic") == 0) { e->spec_self_note = "STOMP_B200_SELF=generic"; return; }
    const char* smode = std::getenv("STOMP_B200_STATES");
    if (smode && std::strcmp(smode, "generic") == 0) { e->spec_self_note = "STOMP_B200_STATES=generic"; return; }
    if (e->self_pairs.n <= 0 || e->self_pairs.n > codegen::kSelfPairCap || e->self_bands.empty()) { e->spec_self_note = "pair list too long for the generated kernel"; return; }
    for (int d = 0; d < e->robot.num_joints; ++d)      // the FP32 bands rest on a bound of the centres that unclamped prismatic values can break
        if (e->robot.joint[d].prismatic) { e->spec_self_note = "prismatic joint"; return; }
    codegen::StateKernelOptions opt = state_kernel_options(e);
    opt.self = &e->self_structure;
    opt.no_tail = true;          // the noise-less rollout of a pair-rule engine is a launch of its own (noiseless_tail_available)
    // the FP32 centres of the spheres that still have partners ahead stay in registers: left alone the dual arm's walk takes
    // 228 of them (8 warps per SM); bounded to 168 (12 warps per SM) a dozen values spill
    opt.rollout_lanes = true;
    opt.min_blocks = 384 / codegen::kStateThreads;
    std::string err;
    e->spec_self = codegen::specialised_state_kernel(e->robot, opt, err);
    e->spec_self_note = e->spec_self ? std::string() : err;
}

// tiles per slab: the slabs of a launch are equally wide (ceil(T / 8) n8 tiles over ceil(T / 104) slabs)
int dmma_tiles_for(int T)
{
    const int ntile = (T + 7) / 8;
    const int nslabs = (ntile + kSlabTilesMax - 1) / kSlabTilesMax;
    const int need = (ntile + nslabs - 1) / nslabs;
    for (int cand : {4, 7, 10, 13})
        if (cand >= need) return cand;
    return kSlabTilesMax;
}

size_t dmma_smem_bytes(int T)
{
    return sizeof(double) * (size_t)dmma_slab_rows(T) * dmma_slab_stride(dmma_tiles_for(T));
}

// Raises a kernel's limit of dynamic shared memory to `bytes`, once per engine: the attribute belongs to the device, and one
// engine is one device.
cudaError_t opt_in_smem(stomp_b200_engine* e, const void* kernel, int bytes)
{
    if (e->smem_opted_in.count(kernel)) return cudaSuccess;
    const cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (err == cudaSuccess) e->smem_opted_in.insert(kernel);
    return err;
}

// The Lt slab of the contraction sampler fits at every T a configuration may have: dmma_slab_rows(T) rows of at most
// kSlabTilesMax n8 tiles, 217,088 B (212 KB) at T = STOMP_B200_MAX_TIME_STEPS = 256.
constexpr int kDmmaSmemOptIn = 225 * 1024;
static_assert(sizeof(double) * dmma_slab_rows(STOMP_B200_MAX_TIME_STEPS) * dmma_slab_stride(kSlabTilesMax) <= kDmmaSmemOptIn,
              "the contraction sampler's Lt slab must fit in shared memory at every trajectory length");

// FP64 tensor-core contraction (DMMA)
template <int kTiles, bool kPhilox>
int launch_sample_dmma_t(stomp_b200_engine* e, const LoopParams& lp)
{
    CUDA_TRY(e, opt_in_smem(e, (const void*)sample_rollouts_dmma_kernel<kTiles, kPhilox>, kDmmaSmemOptIn));
    const long long total_cols = (long long)lp.Q * lp.num_gen * lp.D;
    const int ntiles = (int)((total_cols + 7) / 8);
    const int nslabs = (lp.T + 8 * kTiles - 1) / (8 * kTiles);
    const size_t smem = dmma_smem_bytes(lp.T);
    const int per_sm = smem <= 72 * 1024 ? 3 : (smem <= 110 * 1024 ? 2 : 1);
    dim3 grid(std::max(1, std::min((ntiles + kDmmaWarps - 1) / kDmmaWarps, e->num_sms * per_sm)), nslabs);
    Scope s(e, STOMP_B200_KERNEL_SAMPLE);
    sample_rollouts_dmma_kernel<kTiles, kPhilox><<<grid, kDmmaWarps * 32, smem, e->stream>>>(lp, e->limits, lp.tile_counter);
    return check_launch(e, "sample_rollouts_dmma_kernel");
}

template <bool kPhilox>
int launch_sample_dmma(stomp_b200_engine* e, const LoopParams& lp)
{
    switch (dmma_tiles_for(lp.T)) {
        case 4: return launch_sample_dmma_t<4, kPhilox>(e, lp);
        case 7: return launch_sample_dmma_t<7, kPhilox>(e, lp);
        case 10: return launch_sample_dmma_t<10, kPhilox>(e, lp);
        default: return launch_sample_dmma_t<13, kPhilox>(e, lp);
    }
}

// recurrence sampler (L^-1 is banded); fuse: control-cost sums + n^T R n in the same pass
template <bool kPhilox>
int launch_sample_banded(stomp_b200_engine* e, const LoopParams& lp, bool fuse)
{
    const int band = lp.lband_halfwidth <= 4 ? 4 : 6;
    const void* kernel = band == 4 ? (fuse ? (const void*)sample_rollouts_banded_kernel<4, kPhilox, true> : (const void*)sample_rollouts_banded_kernel<4, kPhilox, false>)
                                   : (fuse ? (const void*)sample_rollouts_banded_kernel<6, kPhilox, true> : (const void*)sample_rollouts_banded_kernel<6, kPhilox, false>);
    const size_t smem = sizeof(double) * banded_sampler_smem_doubles(lp.T, lp.N, band);
    if (smem > 48 * 1024) CUDA_TRY(e, opt_in_smem(e, kernel, 120 * 1024));      // long trajectories: the 32 x T tile passes 48 KB
    const int nkb = (lp.num_gen + 31) / 32;
    Scope s(e, STOMP_B200_KERNEL_SAMPLE);
    void* args[] = {const_cast<LoopParams*>(&lp), &e->limits};
    CUDA_TRY(e, launch_dependent(e, 0, kernel, dim3((unsigned)(nkb * lp.D), (unsigned)lp.Q), dim3(kBandedThreads), smem, e->stream, args));
    return check_launch(e, "sample_rollouts_banded_kernel");
}

enum NoiseMode { kNoisePhilox = 0, kNoiseUnit = 1, kNoiseEpsilon = 2 };

// which control-cost row kernels the operator's shape allows.  kRowsWindow: one rule with Toeplitz interior rows, Toeplitz R
// (or no noise adaptation), even T and N >= 12 — the register-window kernel.  kRowsTile: besides, taps -2 .. +2 and R of half
// bandwidth <= 4 — what the fused sampler and the tile kernel are written for.
enum RowsShape { kRowsGeneric, kRowsWindow, kRowsTile };

RowsShape rows_shape(const stomp_b200_engine* e, const LoopParams& lp)
{
    if (!(lp.st_uniform && (lp.r_toeplitz || !lp.use_noise_adaptation) && e->T % 2 == 0 && e->N >= 12)) return kRowsGeneric;
    if (lp.st_dense[0] != 0.0 || lp.st_dense[6] != 0.0) return kRowsWindow;
    return lp.rband_halfwidth <= 4 ? kRowsTile : kRowsWindow;
}

// eight-rows-per-warp control-cost kernel (kernels.cuh), instantiated for the group counts of the usual T.  Its shared memory
// stays under the default 48 KB: 15,488 B at 14 groups.
// (Capping this grid's residency so that it shares every SM with the state kernel was tried — 32 KB of shared memory per
// one-warp CTA, 7 per SM — and lost: a tile's latency is ~10 us whatever runs beside it, so 3.5 waves of 7 warps took 42 us.
// The two kernels overlap only at their tails.)
template <int kGroups>
void launch_rows_tile(const LoopParams& lp, dim3 grid, cudaStream_t stream)
{
    constexpr size_t smem = sizeof(double) * kTileWarps * 8 * tile_noise_stride(kGroups);
    static_assert(smem <= 48 * 1024, "the tile kernel launches without a shared-memory opt-in");
    if (lp.control_costs) control_rows_tile_kernel<kGroups, true><<<grid, kTileWarps * 32, smem, stream>>>(lp);
    else control_rows_tile_kernel<kGroups, false><<<grid, kTileWarps * 32, smem, stream>>>(lp);
}

// control costs + n^T R n of `rows` (rollout, joint) rows with the kernel of the operator's shape (kRowsTile: the tile kernel
// up to 14 groups, N <= 224, beyond that the register-window kernel for five taps), then the fold of the padding rows into
// the per-time-step costs when they are kept
int launch_rows(stomp_b200_engine* e, const LoopParams& rl, RowsShape shape, int rows, cudaStream_t stream)
{
    const dim3 grid8((rows + 7) / 8, e->Q);     // eight rows per warp (tile kernel) or per CTA (window kernel)
    const int groups = tile_groups(e->N);
    const char* name = "control_rows_tile_kernel";
    if (shape == kRowsTile && groups <= 2) launch_rows_tile<2>(rl, grid8, stream);
    else if (shape == kRowsTile && groups <= 4) launch_rows_tile<4>(rl, grid8, stream);
    else if (shape == kRowsTile && groups <= 7) launch_rows_tile<7>(rl, grid8, stream);
    else if (shape == kRowsTile && groups <= 11) launch_rows_tile<11>(rl, grid8, stream);
    else if (shape == kRowsTile && groups <= 14) launch_rows_tile<14>(rl, grid8, stream);
    else if (shape == kRowsTile) {
        control_rows_fast_kernel<true, true><<<grid8, 256, 0, stream>>>(rl);
        name = "control_rows_fast_kernel<true, true>";
    } else if (shape == kRowsWindow) {
        control_rows_fast_kernel<false, false><<<grid8, 256, 0, stream>>>(rl);
        name = "control_rows_fast_kernel<false, false>";
    } else {
        const size_t row_smem = sizeof(double) * (size_t)kRowWarps * (control_row_x_stride(e->N) + control_row_n_stride(e->T));
        control_rows_kernel<<<dim3((rows + kRowWarps - 1) / kRowWarps, e->Q), kRowWarps * 32, row_smem, stream>>>(rl);
        name = "control_rows_kernel";
    }
    if (int rc = check_launch(e, name)) return rc;
    if (rl.control_costs) {
        fold_control_costs_kernel<<<dim3((rows + 127) / 128, e->Q), 128, 0, stream>>>(rl);
        if (int rc = check_launch(e, "fold_control_costs_kernel")) return rc;
    }
    return 0;
}

codegen::StateKernelOptions state_kernel_options(const stomp_b200_engine* e)
{
    codegen::StateKernelOptions opt;
    opt.wide_index = e->sdf.wide_index != 0;
    // The two bounds below hold for ANY value of a revolute joint, but only inside the limits of a prismatic one — and the
    // noise-less rollout (policy parameters) and stomp_b200_evaluate_states (caller's values) are not clamped to the limits:
    // chains with a prismatic joint keep the index clamps and the saturating conversion.
    bool has_prismatic = false;
    for (int d = 0; d < e->robot.num_joints; ++d) has_prismatic = has_prismatic || e->robot.joint[d].prismatic != 0;
    opt.magic_floor = !has_prismatic && codegen::magic_floor_is_safe(e->robot, e->sdf);
    opt.inside_grid = !has_prismatic && codegen::reach_is_inside_grid(e->robot, e->sdf);
    // links between issuing a link's gathers and comparing them.  With the static spheres out of the walk the 7-joint arm is
    // fastest comparing one link later (16.1 against 16.9 us at lag 2 and 17.7 at lag 0, C3 in the loop; 16.9 / 17.8 / 18.4
    // isolated and flushed), the 14-joint dual arm two links later (41.5 against 44.0 us at lag 1): profiles/r5s_*
    opt.compare_lag = e->robot.num_joints > 8 ? 2 : 1;
    // sines / cosines ahead of the chain walk: measured neutral on the 7-joint arm (15.5 vs 15.6 us at C3), a gain on the
    // 14-joint dual arm (46.8 -> 44.0 us at C5; profiles/r3i_state_kernel_variants*.txt)
    opt.batch_sincos = e->robot.num_joints > 8 ? e->robot.num_joints : 0;
    if (const char* hs = std::getenv("STOMP_B200_STATES_STATIC")) opt.hoist_static = std::atoi(hs) != 0;     // A / B: 0 walks every sphere per state
    return opt;
}

// picks the state kernel once per robot description: the run-time specialised one, or the generic one when
// NVRTC is not available / STOMP_B200_STATES=generic (both are CUDA kernels; spec_note says which and why)
void resolve_state_kernel(stomp_b200_engine* e)
{
    if (e->spec_resolved) return;
    e->spec_resolved = true;
    e->spec = nullptr;
    const char* mode = std::getenv("STOMP_B200_STATES");
    if (mode && std::strcmp(mode, "generic") == 0) { e->spec_note = "STOMP_B200_STATES=generic"; return; }
    std::string err;
    e->spec = codegen::specialised_state_kernel(e->robot, state_kernel_options(e), err);
    e->spec_note = e->spec ? std::string() : err;
    // Largest L1: the walk's SDF gathers want it, and an SM whose split is the sampler's (31 KB of shared memory per CTA)
    // then takes no state CTA until it has drained.  Without the preference, CTAs launched as programmatic dependents of the
    // sampler fill the room beside its CTAs and keep that small-L1 split: 16.9 -> 36 us (profiles/r6a_*).  A hint only.
    if (e->spec && cudaKernelSetAttributeForDevice(e->spec->kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                                   (int)cudaSharedmemCarveoutMaxL1, e->cfg.device) != cudaSuccess)
        (void)cudaGetLastError();
    if (e->spec && e->spec->static_kernel) {
        // Spheres on the axis of a chain's first joint do not move with the state: one thread walks them here, with the
        // statements the state kernel would have issued, and every state starts from that verdict.  Robot, spheres or scene
        // changing resets spec_resolved (set_chain / set_spheres / the SDF setters and builders), which brings us back here;
        // the launch is ordered on the main stream behind the copy or build that produced the grid.
        cudaError_t rc = cudaSuccess;
        if (!e->d_static_hit) {
            rc = cudaMalloc((void**)&e->d_static_hit, sizeof(int32_t));
            if (rc == cudaSuccess) e->allocations.push_back(e->d_static_hit);
        }
        if (rc == cudaSuccess) {
            void* args[] = {&e->robot, &e->sdf, &e->d_static_hit};
            rc = cudaLaunchKernel((const void*)e->spec->static_kernel, dim3(1), dim3(32), args, 0, e->stream);
            e->launch_count++;
        }
        if (rc != cudaSuccess) {
            (void)cudaGetLastError();
            err = std::string("stomp_b200_static_spheres: ") + cudaGetErrorString(rc);
            e->spec = nullptr;
            e->spec_note = err;
        }
    }
    if (!e->spec) {     // still a CUDA kernel, but say so: the generic kernel is ~2x slower
        static bool told = false;
        if (!told) std::fprintf(stderr, "stomp_b200: the specialised state kernel is unavailable, using the generic one: %s\n", err.c_str());
        told = true;
    }
}

// the two arguments of the specialised kernel that come from the engine rather than from the loop: the verdict of the static
// spheres, and the multiplier that replaces idx / T where the host can prove it exact (M = floor(2^32 / T) + 1 has
// M T = 2^32 + r with 0 < r <= T, so umulhi(idx, M) = floor(idx / T + idx r / (T 2^32)) = idx / T whenever idx r < 2^32).
// The static verdict exists once the state kernel is resolved, so that happens here.
void finish_state_args(stomp_b200_engine* e, StateKernelArgs& a)
{
    resolve_state_kernel(e);
    a.static_hit = (e->spec && e->spec->static_kernel) ? e->d_static_hit : nullptr;
    const unsigned long long T = (unsigned long long)std::max(a.T, 0), n = (unsigned long long)std::max(a.num_gen, 0);
    a.t_magic = (T >= 2 && n * T * T < (1ull << 32)) ? (uint32_t)((1ull << 32) / T + 1) : 0u;
}

// the noise-less rollout as a tail of the specialised state kernel (no self-collision pairs, 0 / 1 state costs)
bool noiseless_tail_available(stomp_b200_engine* e)
{
    resolve_state_kernel(e);
    return e->spec != nullptr && e->self_pairs.n == 0 && !e->extras_on;
}

void fill_noiseless_tail(const stomp_b200_engine* e, const LoopParams& lp, double* record, NoiselessTail& nl)
{
    nl.theta = lp.theta_all + kPad; nl.row_stride = lp.N; nl.sumw = lp.sumw; nl.query_stride = (int64_t)lp.D * lp.N;
    nl.state = lp.nl_state; nl.verdict = lp.nl_verdict; nl.valid = lp.nl_valid; nl.sums = record;
    nl.total = lp.nl_total; nl.best = lp.best_cost; nl.old_cost = lp.old_cost; nl.improvement = lp.last_improvement;
    nl.iters = lp.iters_used; nl.stop = lp.stop; nl.counter = e->d_nl_counter; nl.note = lp.note; nl.min_cost_improvement = lp.min_cost_improvement;
}

// ---- the argument blocks of the state passes (StateKernelArgs is filled nowhere else) ----
// the generated rollouts of an iteration; with `tail`, the noise-less rollout owed by the previous iteration rides along
StateKernelArgs rollout_state_args(stomp_b200_engine* e, const LoopParams& lp, bool tail)
{
    StateKernelArgs a{};
    a.rollouts = lp.rollouts; a.state_costs = lp.state_costs; a.verdicts = lp.verdicts; a.validity = lp.validity;
    a.sums = lp.sums; a.s_compact = lp.s_compact; a.stop = lp.stop; a.tile_counter = lp.tile_counter;
    a.timeline = lp.timeline ? lp.timeline + 2 * 1 : nullptr;
    a.T = lp.T; a.D = lp.D; a.slots = lp.slots; a.gslots = lp.gslots; a.sumw = lp.sumw; a.num_gen = lp.num_gen;
    a.gen_offset = lp.gen_offset; a.honour_stop = lp.honour_stop;
    a.row_stride = lp.T; a.rollout_stride = (int64_t)lp.D * lp.T;
    if (tail) fill_noiseless_tail(e, lp, lp.nl_sums, a.nl);
    finish_state_args(e, a);
    return a;
}

// the T noise-less states of the iteration `lp`, read in place from the padded policy rows.  With `tail`: the tail alone (no
// generated rollouts), which also finishes the record the next iteration reads; without: one rollout whose verdicts go to
// nl_state / nl_verdict / nl_valid for noiseless_rollout_kernel
StateKernelArgs noiseless_state_args(stomp_b200_engine* e, const LoopParams& lp, bool tail)
{
    StateKernelArgs a{};
    a.stop = lp.stop; a.T = lp.T; a.D = lp.D; a.slots = 1; a.gslots = 1; a.sumw = lp.sumw; a.honour_stop = lp.honour_stop;
    if (tail) {
        a.timeline = lp.timeline ? lp.timeline + 2 * 5 : nullptr;     // the "noiseless" slot: a launch of its own at a join
        a.num_gen = 0; a.row_stride = lp.T; a.rollout_stride = (int64_t)lp.D * lp.T;
        fill_noiseless_tail(e, lp, e->nl_sums2[e->loop.nl_parity], a.nl);
    } else {
        a.rollouts = lp.theta_all + kPad; a.state_costs = lp.nl_state; a.verdicts = lp.nl_verdict; a.validity = lp.nl_valid;
        a.num_gen = 1; a.row_stride = lp.N; a.rollout_stride = (int64_t)lp.D * lp.N;
    }
    finish_state_args(e, a);
    return a;
}

// the caller's trajectories theta [K][D][T] of stomp_b200_evaluate_states, as one query
StateKernelArgs trajectory_state_args(stomp_b200_engine* e, const double* theta, int K, int T, double* costs, uint8_t* verdicts,
                                      uint8_t* validity)
{
    StateKernelArgs a{};
    a.rollouts = theta; a.state_costs = costs; a.verdicts = verdicts; a.validity = validity;
    a.T = T; a.D = e->D; a.slots = K; a.gslots = 1; a.sumw = 1; a.num_gen = K;
    a.row_stride = T; a.rollout_stride = (int64_t)e->D * T;
    finish_state_args(e, a);
    return a;
}

// One state pass over `queries` queries, with the kernel that serves it: while a pair list is set the generated kernel with
// the pair rule when `sane`, else the list walk with centre storage for the robot's spheres; without one the generated
// world-only kernel when `sane`, else the generic kernel.  `sane`: every joint value is finite with |q| <= 1e6 (the generated
// kernels leave out clamps only such values make redundant).  The grids have codegen::kStateThreads threads per CTA; the
// tail's CTAs come first (state_codegen.hpp).  The caller counts the launch (its profiling Scope, or the noise-less rollout's
// category).
int launch_state_pass(stomp_b200_engine* e, const StateKernelArgs& a, cudaStream_t stream, int queries, int pdl_bit, bool sane)
{
    resolve_state_kernel(e);
    constexpr int bt = codegen::kStateThreads;
    const unsigned tail_blocks = a.nl.theta ? (unsigned)((a.T + bt - 1) / bt) : 0u;
    const dim3 grid((unsigned)(((long long)a.num_gen * a.T + bt - 1) / bt) + tail_blocks, (unsigned)queries), block(bt);
    if (e->self_pairs.n > 0) {
        resolve_self_kernel(e);
        if (e->spec_self && sane) {
            constexpr int tw = bt / 32;      // time steps per CTA when the lanes of a warp are rollouts
            const dim3 lanes_grid((unsigned)((a.num_gen + 31) / 32) * (unsigned)((a.T + tw - 1) / tw), grid.y);
            void* args[] = {(void*)&a, &e->robot, &e->sdf, &e->self_pairs, e->self_bands.data()};
            (void)cudaLaunchKernel((const void*)e->spec_self->kernel, e->spec_self->rollout_lanes ? lanes_grid : grid, block, args, 0, stream);
            return check_launch(e, "stomp_b200_states_specialised (pair rule)");
        }
        const int S = e->robot.num_spheres;
        auto walk = [&](auto simple_kernel, auto kernel) {
            if (e->robot.simple_chain) simple_kernel<<<grid, block, 0, stream>>>(a, e->robot, e->sdf, e->self_pairs);
            else kernel<<<grid, block, 0, stream>>>(a, e->robot, e->sdf, e->self_pairs);
        };
        if (S <= 32) walk(states_self_collision_kernel<32, true>, states_self_collision_kernel<32, false>);
        else if (S <= 64) walk(states_self_collision_kernel<64, true>, states_self_collision_kernel<64, false>);
        else walk(states_self_collision_kernel<STOMP_B200_MAX_SPHERES, true>, states_self_collision_kernel<STOMP_B200_MAX_SPHERES, false>);
        return check_launch(e, "states_self_collision_kernel");
    }
    if (e->spec && sane) {
        void* args[] = {(void*)&a, &e->robot, &e->sdf};
        // Only this kernel may be a programmatic dependent: it is the only state kernel that executes griddepcontrol.wait.
        // Any other, launched that way, could read the stop flag and its joint values before the kernel before it wrote them.
        if (pdl_bit >= 0) (void)launch_dependent(e, pdl_bit, (const void*)e->spec->kernel, grid, block, 0, stream, args);
        else (void)cudaLaunchKernel((const void*)e->spec->kernel, grid, block, args, 0, stream);
        return check_launch(e, "stomp_b200_states_specialised");
    }
    if (e->robot.simple_chain) rollout_states_kernel<true><<<grid, block, 0, stream>>>(a, e->robot, e->sdf);
    else rollout_states_kernel<false><<<grid, block, 0, stream>>>(a, e->robot, e->sdf);
    return check_launch(e, "rollout_states_kernel");
}

// the noise-less rollout of the iteration recorded in e->loop.nl_lp (K10 + the wrapper's stop rule): a state pass over its T states,
// then noiseless_rollout_kernel unless the pass was the tail of the specialised kernel, which finishes the record itself.  On
// the side stream behind everything queued on the main stream so far; on_main_stream: the caller is about to wait for the
// result (a join), nothing is there to overlap with — queue behind the update kernel directly; the cross-stream hand-over
// alone cost 13 us of every isolated iteration
int launch_noiseless(stomp_b200_engine* e, bool on_main_stream)
{
    const LoopParams& lp = e->loop.nl_lp;
    e->loop.nl_deferred = false;
    const bool tail = noiseless_tail_available(e);     // first: resolving may queue the static-sphere kernel on the main stream
    cudaStream_t st = on_main_stream ? e->stream : e->side_stream;
    if (!on_main_stream) {
        CUDA_TRY(e, cudaEventRecord(e->ev_applied, e->stream));
        CUDA_TRY(e, cudaStreamWaitEvent(e->side_stream, e->ev_applied, 0));
    }
    // at a join the tail follows the update kernel on the main stream: as a programmatic dependent its CTAs are resident and
    // waiting when the update kernel's last CTA retires (bit 3 of STOMP_B200_PDL)
    if (int rc = launch_state_pass(e, noiseless_state_args(e, lp, tail), st, e->Q, tail && on_main_stream ? 3 : -1, true)) return rc;
    e->launch_count++;
    e->kernel_launches[STOMP_B200_KERNEL_APPLY]++;
    if (!tail) {
        const size_t smem = sizeof(double) * ((size_t)e->D * e->N + e->T + e->sumw);
        noiseless_rollout_kernel<<<e->Q, 256, smem, st>>>(lp, e->robot, e->sdf, e->extras);
        e->launch_count++;
        if (int rc = check_launch(e, "noiseless_rollout_kernel")) return rc;
    }
    if (!on_main_stream) {
        CUDA_TRY(e, cudaEventRecord(e->ev_noiseless, e->side_stream));
        e->loop.noiseless_pending = true;
    }
    return 0;
}

// The generate stage (K1-K3: sampling; K5, K6: the control costs and n^T R n of the generated rows) in the shape
// generate_shape classifies an iteration into.
enum class Sampler {
    kRecurrence,    // sample_rollouts_banded_kernel through the banded L^-1: on-device noise, or STOMP_B200_SAMPLER=banded
    kContraction,   // sample_rollouts_dmma_kernel with the caller's L: injected epsilon, no band table, or STOMP_B200_SAMPLER=dmma
    kShift,         // shift_rollouts_kernel: injected unit noise
};
enum class RowsWork {
    kNone,          // the fused recurrence sampler left C_d and n^T R n, and no per-time-step control cost is kept
    kStore,         // the fused recurrence sampler left the sums; the row kernel stores only the per-time-step control costs
                    // that read-backs and the per-time-step mode need (rows_mask 0)
    kRows,          // the row kernel computes the control costs and n^T R n
    kProjection,    // project_noise_dmma_kernel, then a row pass for the control costs and one for n^T R n
};
struct GenerateShape {
    Sampler sampler;
    bool philox;            // on-device noise (else the caller's epsilon or unit noise)
    bool fused_rows;        // the recurrence sampler computes the control-cost sums and n^T R n itself
    RowsWork rows;
    RowsShape rows_kind;
    bool overlap;           // the rows run on rows_stream beside the state kernel
};

// Reads the engine only, not an iteration's parameters, so that iterate_async can ask before it builds them.  Projection
// is tested as base.Mproj != nullptr rather than cfg.use_projection: an iteration runs only once the control-cost matrices
// are set (ready_to_solve), and stomp_b200_set_control_cost_matrices sets Mproj exactly when use_projection is on.
GenerateShape generate_shape(const stomp_b200_engine* e, int mode)
{
    const LoopParams& b = e->base;
    GenerateShape g;
    g.philox = mode == kNoisePhilox;
    const bool recurrence = b.Lband != nullptr && (e->sampler_switch == SamplerSwitch::kRecurrence ||
                                                   (g.philox && e->sampler_switch == SamplerSwitch::kDefault));
    g.sampler = mode == kNoiseUnit ? Sampler::kShift : (recurrence ? Sampler::kRecurrence : Sampler::kContraction);
    g.rows_kind = rows_shape(e, b);
    g.fused_rows = g.sampler == Sampler::kRecurrence && !b.Mproj && g.rows_kind == kRowsTile;
    if (b.Mproj) g.rows = RowsWork::kProjection;
    else if (g.fused_rows) g.rows = b.control_costs ? RowsWork::kStore : RowsWork::kNone;
    else g.rows = RowsWork::kRows;
    // the rows and the state costs (K4) are independent of each other (different columns of `sums`) and both latency-bound
    // at < 50 % occupancy: side by side on two streams, serial on the main stream while per-kernel profiling is on
    g.overlap = g.rows != RowsWork::kNone && !e->profiling && e->rows_stream != nullptr;
    return g;
}

// K1-K6 of an iteration in shape g: the padding-only control-cost rows when the policy changed, the sampler, then the rows
// of the generated rollouts.  With g.overlap the rows go to rows_stream and ev_rows marks their end; the caller makes the
// main stream wait for it after the state pass.
int launch_generate_stage(stomp_b200_engine* e, const LoopParams& lp, const GenerateShape& g)
{
    // padding-only rows of the control costs: constants of a solve, needed by the fused sampler and the row kernels
    if (e->loop.edge_dirty && lp.num_rules == 1) {
        edge_rows_kernel<<<e->Q, 64, 0, e->stream>>>(lp);
        e->launch_count++;
        if (int rc = check_launch(e, "edge_rows_kernel")) return rc;
        e->loop.edge_dirty = false;
    }
    switch (g.sampler) {
    case Sampler::kRecurrence:
        if (int rc = g.philox ? launch_sample_banded<true>(e, lp, g.fused_rows) : launch_sample_banded<false>(e, lp, g.fused_rows)) return rc;
        break;
    case Sampler::kContraction:
        if (int rc = g.philox ? launch_sample_dmma<true>(e, lp) : launch_sample_dmma<false>(e, lp)) return rc;
        break;
    case Sampler::kShift: {
        Scope sc(e, STOMP_B200_KERNEL_SAMPLE);
        const int per_query = lp.num_gen * e->D * e->T;
        shift_rollouts_kernel<<<dim3(std::min(1024, (per_query + 255) / 256), e->Q), 256, 0, e->stream>>>(lp, e->limits);
        if (int rc = check_launch(e, "shift_rollouts_kernel")) return rc;
        break;
    }
    }
    if (g.rows == RowsWork::kNone) return 0;
    cudaStream_t rows_stream = g.overlap ? e->rows_stream : e->stream;
    if (g.overlap) {
        CUDA_TRY(e, cudaEventRecord(e->ev_sampled, e->stream));
        CUDA_TRY(e, cudaStreamWaitEvent(rows_stream, e->ev_sampled, 0));
    }
    {
        const int rows = lp.num_gen * e->D;
        Scope sc(e, STOMP_B200_KERNEL_ROWS);
        if (g.rows == RowsWork::kProjection) {
            // M-projection (PolicyImprovement.cpp:421-440): noise_projected_ = M * noise_ for the generated rollouts, then
            // the control costs from parameters_ + noise_projected_ (:812-817) and n^T R n from noise_ (:656-663)
            project_noise_dmma_kernel<<<dim3((rows + 31) / 32, (e->T + 63) / 64, e->Q), 128, 0, rows_stream>>>(lp);
            e->launch_count++;
            if (int rc = check_launch(e, "project_noise_dmma_kernel")) return rc;
            LoopParams cpass = lp; cpass.rows_noise = lp.noise_proj; cpass.rows_mask = 1;
            if (int rc = launch_rows(e, cpass, g.rows_kind, rows, rows_stream)) return rc;
            LoopParams qpass = lp; qpass.rows_noise = lp.noise; qpass.rows_mask = 2; qpass.control_costs = nullptr;
            e->launch_count++;
            if (int rc = launch_rows(e, qpass, g.rows_kind, rows, rows_stream)) return rc;
        } else if (g.rows == RowsWork::kStore) {
            LoopParams store = lp; store.rows_mask = 0;
            if (int rc = launch_rows(e, store, g.rows_kind, rows, rows_stream)) return rc;
        } else if (int rc = launch_rows(e, lp, g.rows_kind, rows, rows_stream)) {
            return rc;
        }
    }
    if (g.overlap) CUDA_TRY(e, cudaEventRecord(e->ev_rows, rows_stream));
    return 0;
}

// The update stage (K7-K9: computeRolloutProbabilities, computeParameterUpdates, updateParameters) takes one of four shapes.
// Every rank of a sharded engine classifies alike: the fields involved are set alike on all ranks.
enum class UpdateShape {
    kPeer,          // rollout sharding over the peer-mapped mailboxes: weights_update_peer_kernel, both exchanges inside
    kFused,         // one GPU, no rollout reuse: weights_update_kernel, one launch
    kPerTimestep,   // per-time-step costs (or forward cumulation): rollout_weights_kernel, the pertimestep kernels, apply_update_kernel
    kSeparate,      // rollout_weights_kernel -> weighted_update_kernel -> apply_update_kernel: the NCCL exchange (which sits
                    // between them), rollout reuse, per-kernel profiling, STOMP_B200_FUSE_WEIGHTS=0
};

// world > 1 implies no rollout reuse (stomp_b200_create), and without reuse buffers no rollout is reused (iterate_body)
UpdateShape update_shape(const stomp_b200_engine* e, int world)
{
    if (e->cfg.use_cumulative_costs != 1) return UpdateShape::kPerTimestep;
    if (!e->fuse_weights_allowed || e->profiling) return UpdateShape::kSeparate;
    if (world > 1) return e->peer_ready ? UpdateShape::kPeer : UpdateShape::kSeparate;
    return e->reuse_possible ? UpdateShape::kSeparate : UpdateShape::kFused;
}

// K7-K9 of an iteration on the main stream, with the exchanges of a sharded engine; sets lp.nchunks, lp.wblocks and
// lp.forward_cumulation, which the noise-less rollout and the read-backs take from lp
int launch_update_stage(stomp_b200_engine* e, LoopParams& lp, UpdateShape shape, int world, bool on_graph)
{
    const stomp_b200_config& c = e->cfg;
    if (world > 1 && !e->comm) return fail(e, STOMP_B200_ERR_NOT_READY, "world_size > 1 needs stomp_b200_comm_init");
    lp.nchunks = std::max(1, (lp.num_local + lp.chunk - 1) / lp.chunk);
    // the chunk's weights and weights * quad, later the column sums and the updated row (apply_update_body)
    const size_t update_smem = sizeof(double) * std::max<size_t>(2 * (size_t)lp.chunk, (size_t)e->T + 2 + (size_t)e->N);
    auto launch_weights = [&]() -> int {
        lp.wblocks = std::max(1, std::min(kWeightBlocksMax, (lp.num_rollouts + kWeightThreads - 1) / kWeightThreads));
        Scope sc(e, STOMP_B200_KERNEL_WEIGHTS);
        rollout_weights_kernel<<<dim3(lp.wblocks, e->D, e->Q), kWeightThreads, 0, e->stream>>>(lp);
        return check_launch(e, "rollout_weights_kernel");
    };
    auto launch_apply = [&](UpdateSums sums) -> int {
        Scope sc(e, STOMP_B200_KERNEL_APPLY);
        apply_update_kernel<<<dim3(e->D, e->Q), 256, sizeof(double) * ((size_t)e->T + 2 + (size_t)e->N), e->stream>>>(lp, sums, lp.nchunks);
        return check_launch(e, "apply_update_kernel");
    };
    switch (shape) {
    case UpdateShape::kPeer: {
        lp.wblocks = 1;
        e->px.epoch = ++e->loop.peer_epoch;
        e->px.epoch_ptr = on_graph ? e->d_counters + 1 : nullptr;
        e->loop.tables_gathered = false;
        Scope sc(e, STOMP_B200_KERNEL_UPDATE);
        void* args[] = {&lp, &e->px};
        CUDA_TRY(e, launch_dependent(e, 2, (const void*)weights_update_peer_kernel, dim3(lp.nchunks * e->D), dim3(kUpdateThreads), update_smem, e->stream, args));
        return check_launch(e, "weights_update_peer_kernel");
    }
    case UpdateShape::kFused: {
        lp.wblocks = 1;
        Scope sc(e, STOMP_B200_KERNEL_UPDATE);
        void* args[] = {&lp};
        CUDA_TRY(e, launch_dependent(e, 2, (const void*)weights_update_kernel, dim3(lp.nchunks, e->D, e->Q), dim3(kUpdateThreads), update_smem, e->stream, args));
        return check_launch(e, "weights_update_kernel");
    }
    case UpdateShape::kPerTimestep: {     // Stomp::setCostCumulation(false): probabilities per time step
        if (int rc = launch_weights()) return rc;
        {
            Scope sc(e, STOMP_B200_KERNEL_UPDATE);
            lp.forward_cumulation = c.use_cumulative_costs == 2 ? 1 : 0;
            if (lp.forward_cumulation) {
                pertimestep_suffix_kernel<<<dim3((lp.num_local * e->D + 127) / 128, e->Q), 128, 0, e->stream>>>(lp);
                if (int rc = check_launch(e, "pertimestep_suffix_kernel")) return rc;
            }
            pertimestep_minmax_kernel<<<dim3(e->D, e->Q), 1024, 0, e->stream>>>(lp);
            if (int rc = check_launch(e, "pertimestep_minmax_kernel")) return rc;
            pertimestep_update_kernel<<<dim3((e->T + 127) / 128, e->D, e->Q), 128, 0, e->stream>>>(lp);
            if (int rc = check_launch(e, "pertimestep_update_kernel")) return rc;
        }
        return launch_apply(kSumsReduced);
    }
    case UpdateShape::kSeparate: {
        const bool nccl = world > 1;
        if (nccl) {     // ---- exchange 1: per-rollout cost scalars (SURVEY.md §8e) ----
            e->loop.tables_gathered = true;
            const size_t count = (size_t)lp.num_gen * e->sumw;
            NCCL_TRY(e, g_nccl.AllGather(lp.sums + (size_t)c.rank * count, lp.sums, count, ncclFloat64, e->comm, e->stream));
        }
        if (int rc = launch_weights()) return rc;
        // the apply step rides on the update kernel's last chunk CTA unless the exchange or per-kernel profiling sits between
        const bool fuse_apply = !nccl && !e->profiling;
        {
            Scope sc(e, STOMP_B200_KERNEL_UPDATE);
            weighted_update_kernel<<<dim3(lp.nchunks, e->D, e->Q), kUpdateThreads, update_smem, e->stream>>>(lp, fuse_apply ? 1 : 0);
            if (int rc = check_launch(e, "weighted_update_kernel")) return rc;
        }
        if (nccl) {     // ---- exchange 2: update rows + adaptation numerators ----
            {
                Scope sc(e, STOMP_B200_KERNEL_UPDATE);
                reduce_partials_kernel<<<dim3(e->D, e->Q), 256, 0, e->stream>>>(lp, lp.nchunks);
                if (int rc = check_launch(e, "reduce_partials_kernel")) return rc;
            }
            const size_t count = (size_t)e->Q * e->D * (e->T + 2);
            NCCL_TRY(e, g_nccl.AllReduce(lp.updbuf, lp.updbuf, count, ncclFloat64, ncclSum, e->comm, e->stream));
        }
        return fuse_apply ? 0 : launch_apply(nccl ? kSumsReduced : kSumsPartials);
    }
    }
    return 0;
}

// PolicyImprovement::generateRollouts bookkeeping (PolicyImprovement.cpp:170-186): the rollouts the next iteration generates,
// in all and on this rank, and the ones it keeps from the last
struct RolloutPlan { int gen, gen_local, reused; };
RolloutPlan plan_rollouts(const stomp_b200_engine* e)
{
    const stomp_b200_config& c = e->cfg;
    const int prev = e->loop.num_rollouts;
    RolloutPlan p;
    p.gen = c.num_rollouts_per_iteration;
    if (prev + p.gen < c.min_rollouts) p.gen = c.min_rollouts - prev;
    p.reused = prev;
    if (prev + p.gen > c.max_rollouts) p.reused = prev - (prev + p.gen - c.max_rollouts);
    if (p.reused < 0) p.reused = 0;
    p.gen_local = p.gen / (c.shard_mode == 0 ? c.world_size : 1);
    return p;
}

int iterate_body(stomp_b200_engine* e, int iteration, int mode, int honour_stop, bool on_graph)
{
    const stomp_b200_config& c = e->cfg;
    const int world = c.shard_mode == 0 ? c.world_size : 1;
    const int prev = e->loop.num_rollouts;
    const auto [gen, gen_local, reused] = plan_rollouts(e);
    if (world > 1 && (reused != 0 || gen % world != 0))
        return fail(e, STOMP_B200_ERR_UNSUPPORTED, "rollout sharding needs min = max = per-iteration rollouts, divisible by world_size");
    if (!e->reuse_possible && reused != 0) return fail(e, STOMP_B200_ERR_UNSUPPORTED, "internal: reuse without reuse buffers");
    int n = reused + gen;
    const bool have_nl = e->loop.noiseless_valid;
    const int nl_gslot = have_nl ? n : -1;
    if (have_nl) ++n;

    LoopParams lp = e->base;
    lp.num_gen = gen_local;
    lp.gen_global = gen;
    lp.gen_offset = (world > 1) ? c.rank * gen_local : 0;
    lp.num_rollouts = n;
    lp.noiseless_slot = have_nl ? gen_local + reused : -1;
    lp.noiseless_gslot = nl_gslot;
    lp.num_local = gen_local + reused + (have_nl ? 1 : 0);
    lp.honour_stop = honour_stop;
    lp.iteration = iteration;
    lp.store_unit = c.keep_debug_tensors;
    lp.counters = on_graph ? e->d_counters : nullptr;
    lp.early_sampler = e->early_sampler ? 1 : 0;
    lp.nl_sums = e->nl_sums2[e->loop.nl_parity];
    lp.nl_sums_next = e->nl_sums2[e->loop.nl_parity ^ 1];
    // the noise-less rollout of the previous iteration: a tail of this iteration's state kernel launch when that kernel is the
    // specialised one, else two kernels on the side stream, under this iteration's sampling and costs
    bool tail_in_state_kernel = false;
    if (e->loop.nl_deferred) {
        if (noiseless_tail_available(e)) { tail_in_state_kernel = true; e->loop.nl_deferred = false; }
        else if (int rc = launch_noiseless(e, false)) return rc;
    }
    if (e->timeline_on) {
        lp.timeline = e->d_timeline + (size_t)(e->timeline_count % kTimelineRing) * kTimelineKernels * 2;
        e->timeline_count++;
    }

    // ---- noise magnitude (Stomp.cpp:179, PolicyImprovement.cpp:162-163) ----
    if (!e->loop.adapted_valid) {
        SigmaIt s;
        for (int d = 0; d < e->D; ++d) s.v[d] = c.noise_stddev[d] * std::pow(c.noise_decay[d], iteration - 1);
        Scope sc(e, STOMP_B200_KERNEL_APPLY);
        set_sigma_by_value_kernel<<<(e->Q * e->D + 127) / 128, 128, 0, e->stream>>>(lp, s);
        if (int rc = check_launch(e, "set_sigma_kernel")) return rc;
    }

    // ---- reused rollouts (PolicyImprovement.cpp:188-255) ----
    if (e->reuse_possible) {
        const int src = e->loop.cur, dst = 1 - e->loop.cur;
        lp.proj = e->proj2[dst]; lp.state_costs = e->state2[dst]; lp.verdicts = e->verdict2[dst];
        if (reused > 0) {
            ReuseParams rp;
            rp.prev = prev; rp.reused = reused; rp.gen = gen_local;
            rp.src_proj = e->proj2[src]; rp.src_state = e->state2[src]; rp.src_verdict = e->verdict2[src];
            rp.src_total = lp.total_cost; rp.order = e->d_order;
            Scope sc(e, STOMP_B200_KERNEL_REUSE);
            reuse_rollouts_kernel<<<e->Q, 256, sizeof(double) * (size_t)prev, e->stream>>>(lp, rp);
            if (int rc = check_launch(e, "reuse_rollouts_kernel")) return rc;
        }
        e->loop.cur = dst;
        e->base.proj = lp.proj; e->base.state_costs = lp.state_costs; e->base.verdicts = lp.verdicts;
    }

    // ---- generate (K1-K6) ----
    const GenerateShape gen_shape = generate_shape(e, mode);
    // the shipped large-K loop (fused sampler, fused weights / update kernel, nothing reads `noise` back): the noise
    // tensor is not materialised — the update kernel subtracts theta from the rollout rows it streams
    const UpdateShape shape = update_shape(e, world);
    const bool one_update_launch = shape == UpdateShape::kFused || shape == UpdateShape::kPeer;
    lp.noise_from_rollouts = (gen_shape.rows == RowsWork::kNone && one_update_launch && !c.keep_debug_tensors && !lp.proj) ? 1 : 0;
    if (int rc = launch_generate_stage(e, lp, gen_shape)) return rc;
    {
        const int states = gen_local * e->T;
        Scope sc(e, STOMP_B200_KERNEL_COST);
        if (int rc = launch_state_pass(e, rollout_state_args(e, lp, tail_in_state_kernel), e->stream, e->Q, 1, true)) return rc;
        if (e->extras_on) {     // alternative state costs: a pass of their own, then S_k in a fixed order
            state_cost_extras_kernel<<<dim3((states + 127) / 128, e->Q), 128, 0, e->stream>>>(lp, e->robot, e->sdf, e->extras);
            if (int rc = check_launch(e, "state_cost_extras_kernel")) return rc;
            state_row_sums_kernel<<<dim3((gen_local + 7) / 8, e->Q), 256, 0, e->stream>>>(lp);
            if (int rc = check_launch(e, "state_row_sums_kernel")) return rc;
            e->launch_count += 2;
        }
    }
    if (gen_shape.overlap) CUDA_TRY(e, cudaStreamWaitEvent(e->stream, e->ev_rows, 0));
    // ---- the noise-less rollout of the previous iteration is needed from here on ----
    if (e->loop.noiseless_pending) {
        CUDA_TRY(e, cudaStreamWaitEvent(e->stream, e->ev_noiseless, 0));
        e->loop.noiseless_pending = false;
    }
    if (reused > 0) {
        const int warps = 8;
        const size_t smem = sizeof(double) * (size_t)warps * (e->N + e->T);
        dim3 grid(std::min(148, (reused * e->D + warps - 1) / warps), e->Q);
        Scope sc(e, STOMP_B200_KERNEL_REUSE);
        reused_control_cost_kernel<<<grid, warps * 32, smem, e->stream>>>(lp, gen_local, reused);
        if (int rc = check_launch(e, "reused_control_cost_kernel")) return rc;
    }

    if (int rc = launch_update_stage(e, lp, shape, world, on_graph)) return rc;
    stomp_b200_engine::LoopState& s = e->loop;
    s.last_wblocks = lp.wblocks;
    s.last_noise_from_rollouts = lp.noise_from_rollouts != 0;
    // ---- noise-less rollout (K10): owed; launched on the side stream by the next iteration or the next join ----
    s.nl_lp = lp;
    s.nl_deferred = true;
    s.nl_parity ^= 1;                             // the record this iteration's update wrote is what the next one reads
    if (on_graph && shape != UpdateShape::kPeer) ++s.peer_epoch;        // the sampler advances counters[1] on every replayed iteration: keep the host's mirror in step

    s.num_rollouts = n;
    s.last_gen = gen_local;
    s.last_local = lp.num_local;
    s.last_noiseless_slot = lp.noiseless_slot;
    s.noiseless_valid = true;
    if (c.use_noise_adaptation) s.adapted_valid = true;
    return 0;
}

__global__ void set_counters_kernel(uint32_t* counters, uint32_t iteration, uint32_t epoch)
{
    counters[0] = iteration;
    counters[1] = epoch;
    counters[2] = iteration;     // the sampler's own copy and its ticket counter (LoopParams::counters)
    counters[3] = 0u;
}

// One Stomp::runSingleIteration for all local queries, queued on the stream (no host synchronisation).  Steady-state
// iterations of the shipped large-K loop — on-device sampler, fused weights / update kernel (single GPU or peer exchange),
// no rollout reuse, nothing per-iteration left in the kernel parameters — are captured ONCE into a CUDA graph with the shape
//     [noise-less rollout of the previous iteration || sampler -> state kernel] -> weights / update
// per (honour_stop, record parity), and replayed with one cudaGraphLaunch: the kernel-to-kernel launch gaps and the host's
// per-launch cost (which bounds a rollout shard of a few hundred rollouts) go away.  The iteration number and the exchange
// epoch are device-side counters then (LoopParams::counters).  Everything else runs iterate_body directly.
int iterate_async(stomp_b200_engine* e, int iteration, int mode, int honour_stop, bool allow_graph = true)
{
    e->scalars_fresh = false; e->solution_fresh = false;
    e->note_writers_in_flight = true;
    const stomp_b200_config& c = e->cfg;
    const int world = c.shard_mode == 0 ? c.world_size : 1;
    const UpdateShape shape = update_shape(e, world);
    const GenerateShape gen_shape = generate_shape(e, mode);
    // nl_deferred: the first iteration after a join (the owed rollout was flushed for the caller) happens once per call, not
    // worth a capture (~0.15 ms) of its own
    bool eligible = allow_graph && e->graphs_allowed && e->d_counters && !e->timeline_on &&
                    e->loop.nl_deferred && e->loop.nl_lp.honour_stop == honour_stop &&
                    gen_shape.philox && gen_shape.sampler == Sampler::kRecurrence && gen_shape.rows != RowsWork::kProjection &&
                    (shape == UpdateShape::kFused || shape == UpdateShape::kPeer) &&
                    e->loop.noiseless_valid && !c.keep_debug_tensors && !e->loop.edge_dirty && !e->extras_on &&
                    !e->loop.noiseless_pending;
    eligible = eligible && noiseless_tail_available(e);      // the side-stream rollout bakes per-iteration state into its parameters
    // A sampler that is launched as a programmatic dependent of the previous iteration's update kernel draws its noise beside
    // it (LoopParams::early_sampler); a graph boundary is a full dependency and would undo that.  On one GPU with a grid that
    // fills it the loop is GPU-bound either way, and plain launches keep the overlap: 50.2 against 58.1 us per C3 iteration
    // (profiles/r5d_early_sampler_ab.txt).  Shards and small problems (no dependent launch of the sampler) keep the graph.
    if (eligible && e->early_sampler && (e->pdl_mask & 1) && !e->graph_over_overlap) {
        const long long sampler_ctas = (long long)((c.num_rollouts_per_iteration / world + 31) / 32) * e->D * e->Q;
        if (sampler_ctas >= 5LL * e->num_sms) eligible = false;
    }
    if (eligible && !e->loop.adapted_valid)     // sigma is a per-iteration kernel parameter unless it does not decay
        for (int d = 0; d < e->D; ++d) eligible = eligible && c.noise_decay[d] == 1.0;
    if (!eligible) return iterate_body(e, iteration, mode, honour_stop, false);
    if (e->streak_epoch != e->config_epoch) { e->streak_epoch = e->config_epoch; e->eligible_streak = 0; }
    if (e->eligible_streak < 2) {               // every kernel of the steady iteration has run before anything is captured
        e->eligible_streak++;
        return iterate_body(e, iteration, mode, honour_stop, false);
    }
    stomp_b200_engine::IterationGraph& g = e->graphs[honour_stop ? 1 : 0][e->loop.nl_parity];
    if (e->dev_iteration_next != iteration || e->dev_epoch_next != (long long)e->loop.peer_epoch) {
        set_counters_kernel<<<1, 1, 0, e->stream>>>(e->d_counters, (uint32_t)iteration, e->loop.peer_epoch);
        e->launch_count++;
        if (int rc = check_launch(e, "set_counters_kernel")) return rc;
    }
    if (!g.exec || g.config_epoch != e->config_epoch) {
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
        const stomp_b200_engine::LoopState loop_before = e->loop;
        const LoopParams base_before = e->base;
        const int64_t launches_before = e->launch_count;
        cudaGraph_t graph = nullptr;
        cudaError_t err = cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal);
        int rc = 0;
        if (err == cudaSuccess) {
            rc = iterate_body(e, iteration, mode, honour_stop, true);
            err = cudaStreamEndCapture(e->stream, &graph);
            if (err == cudaSuccess && rc == 0) err = cudaGraphInstantiate(&g.exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
        }
        if (err != cudaSuccess || rc != 0) {    // no graph on this engine: run the iteration directly from the saved state
            (void)cudaGetLastError();
            if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
            e->loop = loop_before; e->base = base_before; e->launch_count = launches_before;
            e->graphs_allowed = false;
            e->dev_iteration_next = e->dev_epoch_next = -1;
            return iterate_body(e, iteration, mode, honour_stop, false);
        }
        g.config_epoch = e->config_epoch;
        g.launches = e->launch_count - launches_before;
        g.after = e->loop;
    } else {
        // Replay.  The iteration leaves the loop state it left in the capture, but for the exchange epoch and the owed
        // rollout's iteration number, which advance: nl_parity and honour_stop are the graph's key; without rollout reuse
        // (which eligibility implies) `cur` never moves and the rollout record is the same in every iteration; edge_dirty
        // and noiseless_pending are false by eligibility; tables_gathered is false on the peer shape and always true on one
        // GPU; adapted_valid is false without noise adaptation and true after its first iteration with it.
        const uint32_t epoch = e->loop.peer_epoch + 1;
        e->loop = g.after;
        e->loop.peer_epoch = epoch;
        e->loop.nl_lp.iteration = iteration;
        e->launch_count += g.launches;
    }
    CUDA_TRY(e, cudaGraphLaunch(g.exec, e->stream));
    e->graph_launches++;
    e->dev_iteration_next = (long long)iteration + 1;
    e->dev_epoch_next = (long long)e->loop.peer_epoch;
    return 0;
}

// Peer-exchange mode leaves the rollout-indexed tables (sums, probabilities, total costs) rank-local: nothing on the data
// path needs them in full.  Read-backs do, so stomp_b200_get_tensor completes them first — a COLLECTIVE call in that mode
// (every rank asks for the same tensors in the same order; tests and bench.py's parity check do).
int gather_tables_for_readback(stomp_b200_engine* e)
{
    if (e->loop.tables_gathered || !e->comm) return 0;
    const stomp_b200_config& c = e->cfg;
    const size_t gl = (size_t)e->loop.last_gen;
    const LoopParams& b = e->base;
    NCCL_TRY(e, g_nccl.AllGather(b.sums + (size_t)c.rank * gl * e->sumw, b.sums, gl * e->sumw, ncclFloat64, e->comm, e->stream));
    NCCL_TRY(e, g_nccl.AllGather(b.prob + (size_t)c.rank * gl * e->D, b.prob, gl * e->D, ncclFloat64, e->comm, e->stream));
    NCCL_TRY(e, g_nccl.AllGather(b.fprob + (size_t)c.rank * gl * e->D, b.fprob, gl * e->D, ncclFloat64, e->comm, e->stream));
    NCCL_TRY(e, g_nccl.AllGather(b.total_cost + (size_t)c.rank * gl, b.total_cost, gl, ncclFloat64, e->comm, e->stream));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    e->loop.tables_gathered = true;
    return 0;
}

void release_peer_exchange(stomp_b200_engine* e)
{
    for (void* p : e->peer_opened) cudaIpcCloseMemHandle(p);
    e->peer_opened.clear();
    if (e->peer_box_own) cudaFree(e->peer_box_own);
    e->peer_box_own = nullptr;
    e->peer_ready = false;
}

// Maps every rank's mailbox into this process (cudaIpc; the handles travel through one ncclAllGather).  All ranks switch
// to the peer exchange together or not at all: the outcome is agreed with an all-reduce(min).  On any failure the NCCL
// exchange stays in place and exchange_note says why.
int setup_peer_exchange(stomp_b200_engine* e)
{
    const stomp_b200_config& c = e->cfg;
    const int W = c.world_size;
    e->exchange_note = "NCCL all-gather + all-reduce";
    if (const char* x = std::getenv("STOMP_B200_EXCHANGE"))
        if (std::strcmp(x, "nccl") == 0) { e->exchange_note += " (STOMP_B200_EXCHANGE=nccl)"; return 0; }
    if (W > kMaxPeers) { e->exchange_note += " (more than 8 ranks)"; return 0; }
    const size_t bytes = peer_box_bytes(W, e->D, e->T);
    int ok = 1;
    std::string why;
    cudaIpcMemHandle_t mine;
    std::memset(&mine, 0, sizeof mine);
    if (cudaMalloc(&e->peer_box_own, bytes) != cudaSuccess) { ok = 0; why = "cudaMalloc of the mailbox failed"; (void)cudaGetLastError(); }
    if (ok && cudaMemsetAsync(e->peer_box_own, 0, bytes, e->stream) != cudaSuccess) { ok = 0; why = "cudaMemset"; (void)cudaGetLastError(); }
    if (ok && cudaIpcGetMemHandle(&mine, e->peer_box_own) != cudaSuccess) { ok = 0; why = "cudaIpcGetMemHandle failed"; (void)cudaGetLastError(); }
    // handles of all ranks (64 bytes each) + one int32 status per rank
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
    const size_t rec = 64 + 16;
    unsigned char* d_rec = nullptr;
    CUDA_TRY(e, cudaMalloc(&d_rec, rec * W));
    std::vector<unsigned char> h_rec(rec * W, 0);
    std::memcpy(h_rec.data() + rec * c.rank, &mine, 64);
    std::memcpy(h_rec.data() + rec * c.rank + 64, &ok, sizeof(int));
    cudaError_t err = cudaMemcpyAsync(d_rec + rec * c.rank, h_rec.data() + rec * c.rank, rec, cudaMemcpyHostToDevice, e->stream);
    if (err != cudaSuccess) { cudaFree(d_rec); e->last_error = "peer exchange: staging copy failed"; return STOMP_B200_ERR_CUDA; }
    ncclResult_t nr = g_nccl.AllGather(d_rec + rec * c.rank, d_rec, rec, ncclChar, e->comm, e->stream);
    if (nr != ncclSuccess) { cudaFree(d_rec); e->last_error = std::string("peer exchange: ncclAllGather: ") + g_nccl.GetErrorString(nr); return STOMP_B200_ERR_NCCL; }
    err = cudaMemcpyAsync(h_rec.data(), d_rec, rec * W, cudaMemcpyDeviceToHost, e->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    if (err != cudaSuccess) { cudaFree(d_rec); e->last_error = "peer exchange: handle read-back failed"; return STOMP_B200_ERR_CUDA; }
    for (int r = 0; r < W && ok; ++r) {
        int theirs = 0;
        std::memcpy(&theirs, h_rec.data() + rec * r + 64, sizeof(int));
        if (!theirs) { ok = 0; why = "rank " + std::to_string(r) + " could not export its mailbox"; }
    }
    std::memset(&e->px, 0, sizeof(e->px));
    std::memset(&e->extras, 0, sizeof(e->extras));
    for (int r = 0; r < W && ok; ++r) {
        if (r == c.rank) { e->px.box[r] = static_cast<unsigned char*>(e->peer_box_own); continue; }
        cudaIpcMemHandle_t h;
        std::memcpy(&h, h_rec.data() + rec * r, 64);
        void* mapped = nullptr;
        if (cudaIpcOpenMemHandle(&mapped, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            ok = 0; why = std::string("cudaIpcOpenMemHandle of rank ") + std::to_string(r) + ": " + cudaGetErrorString(cudaGetLastError());
        } else {
            e->peer_opened.push_back(mapped);
            e->px.box[r] = static_cast<unsigned char*>(mapped);
        }
    }
    // agreement: min over the ranks of "every mailbox is mapped here"
    int32_t* d_ok = reinterpret_cast<int32_t*>(d_rec);
    int32_t h_ok = ok;
    err = cudaMemcpyAsync(d_ok, &h_ok, sizeof h_ok, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) {
        nr = g_nccl.AllReduce(d_ok, d_ok, 1, ncclInt32, ncclMin, e->comm, e->stream);
        if (nr != ncclSuccess) { cudaFree(d_rec); e->last_error = std::string("peer exchange: ncclAllReduce: ") + g_nccl.GetErrorString(nr); return STOMP_B200_ERR_NCCL; }
        err = cudaMemcpyAsync(&h_ok, d_ok, sizeof h_ok, cudaMemcpyDeviceToHost, e->stream);
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    cudaFree(d_rec);
    if (err != cudaSuccess) { e->last_error = "peer exchange: agreement failed"; return STOMP_B200_ERR_CUDA; }
    if (!h_ok) {
        release_peer_exchange(e);
        e->exchange_note += " (peer mailboxes unavailable: " + (why.empty() ? std::string("another rank failed") : why) + ")";
        return 0;
    }
    e->px.world = W; e->px.rank = c.rank; e->px.epoch = 0; e->px.epoch_ptr = nullptr; e->px.error = e->d_peer_error;
    e->px.D = e->D; e->px.T = e->T;
    e->loop.peer_epoch = 0; e->barrier_ticket = 0;
    e->peer_ready = true;
    e->exchange_note = "peer mailboxes over NVLink (cudaIpc), both exchanges inside weights_update_peer_kernel";
    return 0;
}

int ready_to_solve(stomp_b200_engine* e)
{
    if (!e->have_chain || !e->have_spheres || !e->have_sdf || !e->have_matrices)
        return fail(e, STOMP_B200_ERR_NOT_READY, "chain, spheres, SDF and control-cost matrices must be set first");
    for (int q = 0; q < e->Q; ++q)
        if (!e->have_policy[q]) return fail(e, STOMP_B200_ERR_NOT_READY, "stomp_b200_set_policy missing for a query");
    return 0;
}

int join_side_stream(stomp_b200_engine* e)
{
    if (e->loop.nl_deferred)
        if (int rc = launch_noiseless(e, true)) return rc;
    if (e->loop.noiseless_pending) {
        CUDA_TRY(e, cudaStreamWaitEvent(e->stream, e->ev_noiseless, 0));
        e->loop.noiseless_pending = false;
    }
    return 0;
}

// One read-back per poll: the per-query scalars (one pinned block) and, on request, the solution rows
// parameters_all_[d][6 + t] (StompPlanner.cpp:148-163) into their pinned mirror; one synchronisation for both.
constexpr size_t kSolutionMirrorCap = (size_t)64 << 20;
int fetch_query_scalars(stomp_b200_engine* e, bool with_solution = false)
{
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaMemcpyAsync(e->h_scalars, e->d_scalars, e->scalar_bytes, cudaMemcpyDeviceToHost, e->stream));
    const size_t sol_bytes = sizeof(double) * (size_t)e->Q * e->D * e->T;
    if (with_solution && sol_bytes <= kSolutionMirrorCap) {
        if (!e->h_solution) CUDA_TRY(e, cudaMallocHost(&e->h_solution, sol_bytes));
        CUDA_TRY(e, cudaMemcpy2DAsync(e->h_solution, sizeof(double) * e->T, e->base.theta_all + kPad, sizeof(double) * e->N,
                                      sizeof(double) * e->T, (size_t)e->Q * e->D, cudaMemcpyDeviceToHost, e->stream));
    } else with_solution = false;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    e->note_writers_in_flight = false;
    e->scalars_fresh = true;
    e->solution_fresh = with_solution;
    std::fill(e->policy_in_flight.begin(), e->policy_in_flight.end(), 0);
    resolve_profile(e);
    if (e->peer_ready && *e->h_peer_error != 0)
        return fail(e, STOMP_B200_ERR_NCCL, "peer exchange: a rank did not publish within 4 s (rank missing, or ranks not running the same iterations)");
    return 0;
}

}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

int stomp_b200_abi_version(void) { return STOMP_B200_ABI_VERSION; }

void stomp_b200_default_config(stomp_b200_config* cfg)
{
    if (!cfg) return;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->abi_version = STOMP_B200_ABI_VERSION;
    cfg->num_queries = 1;
    cfg->movement_duration = 5.0;
    cfg->control_cost_weight = 0.001;
    cfg->min_cost_improvement = 0.01;
    for (int d = 0; d < STOMP_B200_MAX_DIMS; ++d) { cfg->noise_stddev[d] = 0.1; cfg->noise_decay[d] = 1.0; cfg->noise_min_stddev[d] = 0.01; }
    cfg->derivative_weights[2] = 1.0;
    cfg->cost_scaling_h = 10.0;
    cfg->use_noise_adaptation = 1;
    cfg->use_cumulative_costs = 1;
    cfg->world_size = 1;
    cfg->seed = 2024;
}

const char* stomp_b200_status_string(int status)
{
    switch (status) {
        case STOMP_B200_OK: return "ok";
        case STOMP_B200_ERR_INVALID_ARGUMENT: return "invalid argument";
        case STOMP_B200_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
        case STOMP_B200_ERR_CUDA: return "CUDA error";
        case STOMP_B200_ERR_NOT_READY: return "engine not ready";
        case STOMP_B200_ERR_UNSUPPORTED: return "not supported by this build";
        case STOMP_B200_ERR_NCCL: return "NCCL error";
        case STOMP_B200_ERR_OUT_OF_MEMORY: return "out of device memory";
        default: return "unknown status";
    }
}

const char* stomp_b200_last_error(const stomp_b200_engine* e) { return e ? e->last_error.c_str() : "null engine"; }

int stomp_b200_create(const stomp_b200_config* cfg, stomp_b200_engine** out)
{
    if (!cfg || !out) return STOMP_B200_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (cfg->abi_version != STOMP_B200_ABI_VERSION) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->num_dimensions < 1 || cfg->num_dimensions > STOMP_B200_MAX_DIMS) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->num_time_steps < 2 || cfg->num_time_steps > STOMP_B200_MAX_TIME_STEPS) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->num_rollouts_per_iteration < 1 || cfg->max_rollouts < cfg->num_rollouts_per_iteration ||
        cfg->min_rollouts > cfg->max_rollouts || cfg->min_rollouts < 1)
        return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->num_queries < 1 || cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size)
        return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->shard_mode != 0 && cfg->shard_mode != 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    const bool reuse_possible = cfg->num_rollouts_per_iteration < cfg->max_rollouts || cfg->min_rollouts > cfg->num_rollouts_per_iteration;
    // Stomp::setCostCumulation(false): built for the plain case (one GPU, no rollout reuse)
    if (cfg->use_cumulative_costs < 0 || cfg->use_cumulative_costs > 2) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (cfg->use_cumulative_costs != 1 && (cfg->world_size > 1 || reuse_possible)) return STOMP_B200_ERR_UNSUPPORTED;
    if (cfg->shard_mode == 0 && cfg->world_size > 1 && cfg->num_queries != 1) return STOMP_B200_ERR_UNSUPPORTED;
    // rollout sharding: every rank draws the same number of rollouts every iteration, and none is reused
    if (cfg->shard_mode == 0 && cfg->world_size > 1 && (reuse_possible || cfg->num_rollouts_per_iteration % cfg->world_size != 0))
        return STOMP_B200_ERR_UNSUPPORTED;

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return STOMP_B200_ERR_NO_DEVICE;
    if (cfg->device < 0 || cfg->device >= ndev) return STOMP_B200_ERR_INVALID_ARGUMENT;

    stomp_b200_engine* e = new stomp_b200_engine();
    e->cfg = *cfg;
    e->T = cfg->num_time_steps; e->D = cfg->num_dimensions; e->N = e->T + 2 * kPad;
    e->sumw = 1 + 3 * e->D;
    if (cfg->shard_mode == 1 && cfg->world_size > 1) {
        // balanced contiguous blocks: floor(Q / G) queries per rank, the first Q mod G ranks one more (no rank is left
        // empty as long as Q >= G; ceil-sized blocks left the last of 8 ranks without work at Q = 25)
        const int per = cfg->num_queries / cfg->world_size, rem = cfg->num_queries % cfg->world_size;
        e->query_offset = cfg->rank * per + std::min(cfg->rank, rem);
        e->Q = per + (cfg->rank < rem ? 1 : 0);
        if (e->Q == 0) { delete e; return STOMP_B200_ERR_INVALID_ARGUMENT; }
    } else {
        e->Q = cfg->num_queries;
    }
    const int world = cfg->shard_mode == 0 ? cfg->world_size : 1;
    e->reuse_possible = reuse_possible;
    e->gslots = cfg->max_rollouts + 1;
    e->slots = (world > 1 ? cfg->max_rollouts / world : cfg->max_rollouts) + 1;
    e->have_policy.assign(e->Q, 0);

#define CREATE_TRY(call)                       \
    do {                                       \
        int _rc = (call);                      \
        if (_rc != 0) {                        \
            stomp_b200_destroy(e);             \
            return _rc;                        \
        }                                      \
    } while (0)
#define CREATE_CUDA(call)                                                          \
    do {                                                                           \
        cudaError_t _err = (call);                                                 \
        if (_err != cudaSuccess) {                                                 \
            std::fprintf(stderr, "stomp_b200_create: %s: %s\n", #call, cudaGetErrorString(_err)); \
            stomp_b200_destroy(e);                                                 \
            return STOMP_B200_ERR_CUDA;                                            \
        }                                                                          \
    } while (0)

    CREATE_CUDA(cudaSetDevice(cfg->device));
    CREATE_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaStreamCreateWithFlags(&e->side_stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaEventCreateWithFlags(&e->ev_applied, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&e->ev_noiseless, cudaEventDisableTiming));
    CREATE_CUDA(cudaStreamCreateWithFlags(&e->rows_stream, cudaStreamNonBlocking));
    CREATE_CUDA(cudaEventCreateWithFlags(&e->ev_sampled, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&e->ev_rows, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreate(&e->timer_a));
    CREATE_CUDA(cudaEventCreate(&e->timer_b));

    const size_t Q = e->Q, T = e->T, D = e->D, N = e->N, S = e->slots, GS = e->gslots;
    LoopParams& b = e->base;
    std::memset(&b, 0, sizeof(b));
    b.T = e->T; b.D = e->D; b.N = e->N; b.Q = e->Q; b.slots = e->slots; b.gslots = e->gslots; b.sumw = e->sumw;
    b.query_offset = e->query_offset;
    b.control_cost_weight = cfg->control_cost_weight;
    b.dt = cfg->movement_duration / (cfg->num_time_steps + 1);
    b.cost_scaling_h = cfg->cost_scaling_h;
    b.min_cost_improvement = cfg->min_cost_improvement;
    b.use_noise_adaptation = cfg->use_noise_adaptation;
    b.seed = cfg->seed;
    b.noiseless_slot = -1;

    double* tmp = nullptr;
    CREATE_TRY(dev_alloc(e, &b.theta_all, Q * D * N));
    CREATE_TRY(dev_alloc(e, &tmp, Q * D * T)); b.mincc = tmp;
    CREATE_TRY(dev_alloc(e, &b.rollouts, Q * S * D * T));
    CREATE_TRY(dev_alloc(e, &b.noise, Q * S * D * T));
    b.rows_noise = b.noise;
    b.rows_mask = 3;
    b.per_timestep_minmax = cfg->per_timestep_minmax ? 1 : 0;
    if (cfg->use_projection) {
        CREATE_TRY(dev_alloc(e, &b.noise_proj, Q * S * D * T));
        CREATE_TRY(dev_alloc(e, &e->d_Mproj, T * T));
        CREATE_TRY(dev_alloc(e, &e->d_Minv, T * T));
        // Mproj / Minv stay null in `base` until stomp_b200_set_control_cost_matrices has filled them
    }
    for (int i = 0; i < (e->reuse_possible ? 2 : 1); ++i) {
        CREATE_TRY(dev_alloc(e, &e->state2[i], Q * S * T));
        CREATE_TRY(dev_alloc(e, &e->verdict2[i], Q * S * T));
        if (e->reuse_possible) CREATE_TRY(dev_alloc(e, &e->proj2[i], Q * S * D * T));
    }
    b.state_costs = e->state2[0]; b.verdicts = e->verdict2[0]; b.proj = e->proj2[0];
    CREATE_TRY(dev_alloc(e, &b.validity, Q * S));
    if (cfg->keep_debug_tensors || cfg->use_cumulative_costs != 1) CREATE_TRY(dev_alloc(e, &b.control_costs, Q * S * D * T));
    if (cfg->use_cumulative_costs == 2) CREATE_TRY(dev_alloc(e, &b.pt_cum, Q * S * D * T));
    if (cfg->use_cumulative_costs != 1) {
        CREATE_TRY(dev_alloc(e, &b.pt_prob, Q * GS * D * T));
        CREATE_TRY(dev_alloc(e, &b.pt_minden, Q * D * 2));
    }
    CREATE_TRY(dev_alloc(e, &b.sums, Q * GS * e->sumw));
    CREATE_TRY(dev_alloc(e, &b.total_cost, Q * GS));
    CREATE_TRY(dev_alloc(e, &b.prob, Q * GS * D));
    CREATE_TRY(dev_alloc(e, &b.fprob, Q * GS * D));
    CREATE_TRY(dev_alloc(e, &b.fprob_sum, Q * D));
    CREATE_TRY(dev_alloc(e, &b.sigma, Q * D));
    CREATE_TRY(dev_alloc(e, &b.coef, Q * D * 3));
    CREATE_TRY(dev_alloc(e, &b.updbuf, Q * D * (T + 2)));
    CREATE_TRY(dev_alloc(e, &b.updates, Q * D * T));
    const size_t gen_cap = (size_t)std::max(cfg->num_rollouts_per_iteration, cfg->min_rollouts) / world + 1;
    CREATE_TRY(dev_alloc(e, &b.unit_noise, Q * gen_cap * D * T));
    CREATE_TRY(dev_alloc(e, &b.epsilon, Q * gen_cap * D * T));
    CREATE_TRY(dev_alloc(e, &b.nl_state, Q * T));
    CREATE_TRY(dev_alloc(e, &b.nl_verdict, Q * T));
    CREATE_TRY(dev_alloc(e, &b.nl_control, Q * D * T));
    CREATE_TRY(dev_alloc(e, &e->nl_sums2[0], Q * e->sumw));
    CREATE_TRY(dev_alloc(e, &e->nl_sums2[1], Q * e->sumw));
    CREATE_TRY(dev_alloc(e, &e->d_nl_counter, Q));
    b.nl_sums = e->nl_sums2[0]; b.nl_sums_next = e->nl_sums2[1];
    {
        // the per-query scalars the host reads back live in ONE device block, mirrored by one pinned block: a single
        // D2H copy per read-back.  Layout: [Q] nl_total | [Q] last_improvement | [Q] stop | [Q] iters_used | [Q] nl_valid
        const size_t per_query_bytes = Q * (2 * sizeof(double) + 2 * sizeof(int32_t) + 1);
        const size_t err_off = (per_query_bytes + 7) & ~(size_t)7;           // int32 flag of the peer exchange, after the per-query block
        e->scalar_bytes = err_off + sizeof(int32_t);
        unsigned char* blk = nullptr;
        CREATE_TRY(dev_alloc(e, &blk, e->scalar_bytes + 16));
        e->d_scalars = blk;
        e->d_peer_error = reinterpret_cast<int32_t*>(blk + err_off);
        b.nl_total = reinterpret_cast<double*>(blk);
        b.last_improvement = b.nl_total + Q;
        b.stop = reinterpret_cast<int32_t*>(b.last_improvement + Q);
        b.iters_used = b.stop + Q;
        b.nl_valid = reinterpret_cast<uint8_t*>(b.iters_used + Q);
    }
    CREATE_TRY(dev_alloc(e, &b.old_cost, Q));
    CREATE_TRY(dev_alloc(e, &b.best_cost, Q));
    CREATE_TRY(dev_alloc(e, &e->d_order, Q * S));
    // rollouts per CTA of the weights / update kernels: the kernels are latency chains (cost scan -> exp -> stream of the
    // chunk's rows -> last-CTA reduction), so shorter chunks finish sooner — as long as the grid stays ONE wave (three
    // 256-thread CTAs per SM at 80 registers).  Measured at K = 4096 on one GPU: 128 -> 14.2 us (231 CTAs), 64 -> 15.4 us
    // (455 CTAs: a second wave), 32 -> 24.6 us; a rollout shard of 2048 / 512 rollouts gets 64 / 32.
    {
        cudaDeviceProp prop;
        CREATE_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
        e->num_sms = prop.multiProcessorCount;
        int chunk = 128;
        while (chunk > 32 && (long long)((S + chunk / 2 - 1) / (chunk / 2)) * (long long)D * (long long)Q <= 3LL * e->num_sms) chunk /= 2;
        b.chunk = chunk;
    }
    e->max_chunks = (int)((S + b.chunk - 1) / b.chunk);
    CREATE_TRY(dev_alloc(e, &b.partial, Q * e->max_chunks * D * (T + 2)));
    b.wblocks_cap = (int)((GS + 255) / 256);
    CREATE_TRY(dev_alloc(e, &b.wpart, Q * D * b.wblocks_cap));
    CREATE_TRY(dev_alloc(e, &b.edge_cost, Q * D * 6));
    CREATE_TRY(dev_alloc(e, &b.done_counter, Q * D));
    CREATE_TRY(dev_alloc(e, &b.s_compact, Q * GS));
    CREATE_TRY(dev_alloc(e, &b.c_compact, Q * D * GS));
    CREATE_TRY(dev_alloc(e, &b.tile_counter, 4));
    CREATE_TRY(dev_alloc(e, &e->d_counters, 4));
    if (const char* gr = std::getenv("STOMP_B200_GRAPH")) { e->graphs_allowed = std::strcmp(gr, "0") != 0; e->graph_over_overlap = std::strcmp(gr, "2") == 0; }
    if (const char* pd = std::getenv("STOMP_B200_PDL")) e->pdl_mask = std::atoi(pd) & 15;
    if (const char* es = std::getenv("STOMP_B200_SAMPLER_EARLY")) e->early_sampler = std::strcmp(es, "0") != 0;
    CREATE_TRY(dev_alloc(e, &e->d_timeline, (size_t)kTimelineRing * kTimelineKernels * 2));
    b.world_size = world;

    // control-cost operator: banded differentiation matrices of the active rules (StompUtils.cpp:6-23)
    {
        std::vector<double> band((size_t)kMaxRules * N * 7, 0.0);
        b.num_rules = 0;
        for (int r = 0; r < kMaxRules; ++r) {
            host::DiffBand db = host::differentiation_band(e->N, r, b.dt);
            std::copy(db.c.begin(), db.c.end(), band.begin() + (size_t)r * N * 7);
            if (cfg->derivative_weights[r] != 0.0) {
                b.rule_id[b.num_rules] = r;
                b.rule_sqrt_w[b.num_rules] = std::sqrt(cfg->derivative_weights[r]);
                b.num_rules++;
            }
        }
        b.st_uniform = b.num_rules == 1 && e->N >= 8;
        if (b.st_uniform) std::copy_n(band.data() + ((size_t)b.rule_id[0] * N + 3) * 7, 7, b.st_dense);   // any interior row
        CREATE_TRY(dev_alloc(e, &tmp, band.size())); b.diff_band = tmp;
        CREATE_CUDA(cudaMemcpyAsync(tmp, band.data(), sizeof(double) * band.size(), cudaMemcpyHostToDevice, e->stream));
        CREATE_TRY(dev_alloc(e, &tmp, D)); b.min_stddev = tmp;
        CREATE_CUDA(cudaMemcpyAsync(tmp, cfg->noise_min_stddev, sizeof(double) * D, cudaMemcpyHostToDevice, e->stream));
        CREATE_TRY(dev_alloc(e, &tmp, T * T)); b.Lt = tmp;
        CREATE_TRY(dev_alloc(e, &e->d_Lband, T * 8));
        CREATE_TRY(dev_alloc(e, &tmp, T * (2 * kRBand + 1))); b.Rband = tmp;
        CREATE_CUDA(cudaStreamSynchronize(e->stream));
    }
    CREATE_CUDA(cudaMallocHost(&e->h_scalars, e->scalar_bytes + 16));
    e->h_cost = reinterpret_cast<double*>(e->h_scalars);
    e->h_impr = e->h_cost + Q;
    e->h_stop = reinterpret_cast<int32_t*>(e->h_impr + Q);
    e->h_iters = e->h_stop + Q;
    e->h_valid = reinterpret_cast<uint8_t*>(e->h_iters + Q);
    e->h_peer_error = reinterpret_cast<int32_t*>(e->h_scalars + (e->scalar_bytes - sizeof(int32_t)));
    *e->h_peer_error = 0;
    {
        void* note = nullptr;
        CREATE_CUDA(cudaHostAlloc(&note, sizeof(int32_t) * 2 * Q, cudaHostAllocMapped));
        std::memset(note, 0, sizeof(int32_t) * 2 * Q);
        e->h_note = static_cast<volatile int32_t*>(note);
        void* dnote = nullptr;
        CREATE_CUDA(cudaHostGetDevicePointer(&dnote, note, 0));
        e->base.note = static_cast<int32_t*>(dnote);
        if (const char* s = std::getenv("STOMP_B200_SOLVE_AHEAD")) e->solve_ahead = std::max(0, std::min(16, std::atoi(s)));
        e->policy_in_flight.assign(Q, 0);
        CREATE_CUDA(cudaEventCreateWithFlags(&e->ev_policy, cudaEventDisableTiming));
    }
    std::memset(&e->px, 0, sizeof(e->px));
    {
        cudaDeviceProp prop;
        CREATE_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
        e->num_sms = prop.multiProcessorCount;
    }
    if (const char* s = std::getenv("STOMP_B200_SAMPLER")) {
        if (std::strcmp(s, "dmma") == 0) e->sampler_switch = SamplerSwitch::kContraction;
        else if (std::strcmp(s, "banded") == 0) e->sampler_switch = SamplerSwitch::kRecurrence;
    }
    CREATE_CUDA(cudaFuncSetAttribute(noiseless_rollout_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CREATE_CUDA(cudaFuncSetAttribute(reuse_rollouts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    if (const char* f = std::getenv("STOMP_B200_FUSE_WEIGHTS")) e->fuse_weights_allowed = std::strcmp(f, "0") != 0;
    std::memset(&e->robot, 0, sizeof(e->robot));
    std::memset(&e->sdf, 0, sizeof(e->sdf));
    CREATE_CUDA(cudaStreamSynchronize(e->stream));
#undef CREATE_TRY
#undef CREATE_CUDA
    *out = e;
    return STOMP_B200_OK;
}

int stomp_b200_destroy(stomp_b200_engine* e)
{
    if (!e) return STOMP_B200_OK;
    cudaSetDevice(e->cfg.device);
    if (e->side_stream) cudaStreamSynchronize(e->side_stream);
    if (e->rows_stream) cudaStreamSynchronize(e->rows_stream);
    if (e->stream) cudaStreamSynchronize(e->stream);
    resolve_profile(e);
    for (auto& row : e->graphs)
        for (auto& g : row)
            if (g.exec) cudaGraphExecDestroy(g.exec);
    release_peer_exchange(e);
    if (e->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
    for (void* p : e->allocations) cudaFree(p);
    if (e->d_sdf) cudaFree(e->d_sdf);
    for (void* p : e->self_pair_buffers) cudaFree(p);
    if (e->eval_theta) cudaFree(e->eval_theta);
    if (e->eval_cost) cudaFree(e->eval_cost);
    if (e->eval_verdict) cudaFree(e->eval_verdict);
    if (e->eval_valid) cudaFree(e->eval_valid);
    if (e->h_scalars) cudaFreeHost(e->h_scalars);
    if (e->h_note) cudaFreeHost(const_cast<int32_t*>(e->h_note));
    if (e->h_solution) cudaFreeHost(e->h_solution);
    if (e->h_policy) cudaFreeHost(e->h_policy);
    if (e->ev_policy) cudaEventDestroy(e->ev_policy);
    if (e->timer_a) cudaEventDestroy(e->timer_a);
    if (e->timer_b) cudaEventDestroy(e->timer_b);
    if (e->ev_applied) cudaEventDestroy(e->ev_applied);
    if (e->ev_noiseless) cudaEventDestroy(e->ev_noiseless);
    if (e->side_stream) cudaStreamDestroy(e->side_stream);
    if (e->ev_sampled) cudaEventDestroy(e->ev_sampled);
    if (e->ev_rows) cudaEventDestroy(e->ev_rows);
    if (e->rows_stream) cudaStreamDestroy(e->rows_stream);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return STOMP_B200_OK;
}

// fixed rotation of a URDF joint origin: Rz(yaw) * Ry(pitch) * Rx(roll)
static void rpy_matrix(const double rpy[3], double A[9])
{
    double sr, cr, sp, cp, sy, cy;
    det_sincos(rpy[0], sr, cr);
    det_sincos(rpy[1], sp, cp);
    det_sincos(rpy[2], sy, cy);
    A[0] = cy * cp; A[1] = cy * sp * sr - sy * cr; A[2] = cy * sp * cr + sy * sr;
    A[3] = sy * cp; A[4] = sy * sp * sr + cy * cr; A[5] = sy * sp * cr - cy * sr;
    A[6] = -sp;     A[7] = cp * sr;                A[8] = cp * cr;
}

int stomp_b200_set_chain(stomp_b200_engine* e, int32_t num_joints, const double* origin_xyz, const double* origin_rpy,
                         const double* axis, const int32_t* parent, const int32_t* prismatic, const double* lower,
                         const double* upper)
{
    if (!e || !origin_xyz || !origin_rpy || !axis || !lower || !upper) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (num_joints != e->D) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "num_joints != num_dimensions");
    RobotParams& r = e->robot;
    r.num_joints = num_joints;
    for (int d = 0; d < num_joints; ++d) {
        JointParams& j = r.joint[d];
        j.parent = parent ? parent[d] : (d == 0 ? -1 : d - 1);
        if (!(j.parent == -1 || j.parent == d - 1))
            return fail(e, STOMP_B200_ERR_UNSUPPORTED, "parent[d] must be d-1 or -1 (serial chains, restartable)");
        j.prismatic = prismatic ? prismatic[d] : 0;
        const double* a = axis + 3 * d;
        j.o_mask = 0;
        for (int i = 0; i < 3; ++i) {
            j.o[i] = origin_xyz[3 * d + i];
            j.axis[i] = a[i];
            if (j.o[i] != 0.0) j.o_mask |= 1 << i;
        }
        const double* rpy = origin_rpy + 3 * d;
        j.fixed_rot_identity = (rpy[0] == 0.0 && rpy[1] == 0.0 && rpy[2] == 0.0) ? 1 : 0;
        rpy_matrix(rpy, j.A);
        if (j.fixed_rot_identity) { j.A[0] = j.A[4] = j.A[8] = 1.0; j.A[1] = j.A[2] = j.A[3] = j.A[5] = j.A[6] = j.A[7] = 0.0; }
        int kind = kAxisGeneral;
        if (a[1] == 0.0 && a[2] == 0.0 && a[0] == 1.0) kind = kAxisX;
        else if (a[0] == 0.0 && a[2] == 0.0 && a[1] == 1.0) kind = kAxisY;
        else if (a[0] == 0.0 && a[1] == 0.0 && a[2] == 1.0) kind = kAxisZ;
        else if (a[1] == 0.0 && a[2] == 0.0 && a[0] == -1.0) kind = kAxisNegX;
        else if (a[0] == 0.0 && a[2] == 0.0 && a[1] == -1.0) kind = kAxisNegY;
        else if (a[0] == 0.0 && a[1] == 0.0 && a[2] == -1.0) kind = kAxisNegZ;
        j.axis_kind = kind;
        r.lower[d] = lower[d];
        r.upper[d] = upper[d];
        e->limits.lower[d] = lower[d];
        e->limits.upper[d] = upper[d];
    }
    r.simple_chain = 1;
    for (int d = 0; d < num_joints; ++d)
        if (r.joint[d].prismatic || !r.joint[d].fixed_rot_identity || r.joint[d].axis_kind == kAxisGeneral) r.simple_chain = 0;
    e->have_chain = true;
    e->spec_resolved = false;
    e->config_epoch++;
    return STOMP_B200_OK;
}

// smallest binary32 >= r (SphereParams::r_up)
static float float_at_or_above(double r)
{
    float f = (float)r;                       // round to nearest
    if ((double)f < r) {                      // step up one ulp
        uint32_t u;
        std::memcpy(&u, &f, sizeof u);
        if (f == 0.0f) u = 1u;                // smallest subnormal
        else if (f > 0.0f) u += 1u;
        else u -= 1u;
        std::memcpy(&f, &u, sizeof u);
    }
    return f;
}

int stomp_b200_set_spheres(stomp_b200_engine* e, int32_t num_spheres, const int32_t* link, const double* centre_xyz,
                           const double* radius)
{
    if (!e || !link || !centre_xyz || !radius) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (num_spheres < 1 || num_spheres > STOMP_B200_MAX_SPHERES) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "sphere count out of range");
    RobotParams& r = e->robot;
    r.num_spheres = num_spheres;
    for (int d = 0; d <= STOMP_B200_MAX_DIMS; ++d) r.sphere_begin[d] = 0;
    for (int s = 0; s < num_spheres; ++s) {
        if (link[s] < 0 || link[s] >= e->D) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "sphere link out of range");
        if (s > 0 && link[s] < link[s - 1]) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "spheres must be sorted by link");
        r.sphere[s].mask = 0;
        for (int i = 0; i < 3; ++i) {
            r.sphere[s].l[i] = centre_xyz[3 * s + i];
            if (r.sphere[s].l[i] != 0.0) r.sphere[s].mask |= 1 << i;
        }
        r.sphere[s].r = radius[s];
        r.sphere[s].r_up = float_at_or_above(radius[s]);
        r.sphere_begin[link[s] + 1] = s + 1;
    }
    for (int d = 1; d <= STOMP_B200_MAX_DIMS; ++d) r.sphere_begin[d] = std::max(r.sphere_begin[d], r.sphere_begin[d - 1]);
    e->have_spheres = true;
    e->spec_resolved = false;
    e->config_epoch++;
    e->self_pairs.n = 0;   // indices and radii of an earlier pair list no longer apply
    e->spec_self = nullptr; e->spec_self_resolved = false; e->self_bands.clear();
    return STOMP_B200_OK;
}

int stomp_b200_set_cost_extras(stomp_b200_engine* e, int32_t use_smooth_cost, double smooth_margin, double smooth_weight,
                               int32_t use_joint_constraint, const double* value, const double* tolerance, double joint_constraint_weight)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (use_joint_constraint && (!value || !tolerance)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "joint constraint needs value and tolerance");
    if (use_smooth_cost && !(smooth_margin >= 0.0 && smooth_weight >= 0.0)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "smooth cost: margin and weight must be >= 0");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    std::memset(&e->extras, 0, sizeof(e->extras));
    e->extras.smooth = use_smooth_cost ? 1 : 0;
    e->extras.smooth_margin = smooth_margin;
    e->extras.smooth_weight = smooth_weight;
    e->extras.joint_constraint = use_joint_constraint ? 1 : 0;
    e->extras.jc_weight = joint_constraint_weight;
    for (int d = 0; d < e->D && use_joint_constraint; ++d) {
        if (!(std::fabs(value[d]) <= 1e6) || !(tolerance[d] >= 0.0)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "joint constraint: bad value or tolerance");
        e->extras.jc_value[d] = value[d];
        e->extras.jc_tolerance[d] = tolerance[d];
    }
    e->extras_on = use_smooth_cost || use_joint_constraint;
    e->config_epoch++;
    return STOMP_B200_OK;
}

int stomp_b200_set_self_collision(stomp_b200_engine* e, int32_t num_pairs, const int32_t* pairs)
{
    if (!e || num_pairs < 0 || (num_pairs > 0 && !pairs)) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_spheres) return fail(e, STOMP_B200_ERR_NOT_READY, "stomp_b200_set_spheres comes first");
    const RobotParams& r = e->robot;
    const int S = r.num_spheres, D = e->D;
    e->config_epoch++;
    if (num_pairs > S * (S - 1) / 2) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "more pairs than distinct sphere pairs");
    std::vector<int> link_of((size_t)S, 0);
    for (int d = 0; d < D; ++d)
        for (int s = r.sphere_begin[d]; s < r.sphere_begin[d + 1]; ++s) link_of[s] = d;
    std::vector<int2> ij((size_t)num_pairs);
    for (int p = 0; p < num_pairs; ++p) {
        int i = pairs[2 * p], j = pairs[2 * p + 1];
        if (i > j) std::swap(i, j);
        if (i < 0 || j >= S || i == j) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "self-collision pair: sphere index out of range");
        ij[p] = make_int2(i, j);
    }
    // blocks by link pair (spheres are sorted by link, so link_of is monotone in the sphere index)
    std::stable_sort(ij.begin(), ij.end(), [&](const int2& u, const int2& v) {
        return std::make_pair(link_of[u.x], link_of[u.y]) < std::make_pair(link_of[v.x], link_of[v.y]);
    });
    std::vector<double> limit2((size_t)num_pairs);
    for (int p = 0; p < num_pairs; ++p) {
        const double sum = r.sphere[ij[p].x].r + r.sphere[ij[p].y].r;
        limit2[p] = sum * sum;
    }
    // one bounding sphere per link around its collision spheres, in the link frame; the radius is inflated (1e-9 relative +
    // 1e-9 m) — orders of magnitude above the rounding of the centres, so the cull is conservative
    std::vector<double> bound(4 * (size_t)D, 0.0), bound_radius((size_t)D, 0.0);
    for (int d = 0; d < D; ++d) {
        const int s0 = r.sphere_begin[d], s1 = r.sphere_begin[d + 1];
        if (s1 <= s0) continue;
        for (int i = 0; i < 3; ++i) {
            double m = 0.0;
            for (int s = s0; s < s1; ++s) m += r.sphere[s].l[i];
            bound[4 * d + i] = m / (s1 - s0);
        }
        double radius = 0.0;
        for (int s = s0; s < s1; ++s) {
            double d2 = 0.0;
            for (int i = 0; i < 3; ++i) { const double t = r.sphere[s].l[i] - bound[4 * d + i]; d2 += t * t; }
            radius = std::max(radius, std::sqrt(d2) + r.sphere[s].r);
        }
        bound_radius[d] = radius * (1.0 + 1e-9) + 1e-9;
    }
    std::vector<int4> block;
    std::vector<double> block_limit2;
    for (int p = 0; p < num_pairs; ++p) {
        const int la = link_of[ij[p].x], lb = link_of[ij[p].y];
        if (block.empty() || block.back().x != la || block.back().y != lb) {
            block.push_back(make_int4(la, lb, p, p));
            const double sum = bound_radius[la] + bound_radius[lb];
            block_limit2.push_back(sum * sum);
        }
        block.back().w = p + 1;
    }
    // ---- the same rule for the generated kernel: FP32 centres in registers, thresholds conservative on both sides ----
    e->spec_self = nullptr; e->spec_self_resolved = false;
    e->self_structure = codegen::SelfPairStructure();
    e->self_bands.clear();
    if (num_pairs > 0 && num_pairs <= codegen::kSelfPairCap) {
        // B bounds |coordinate| of any sphere centre (chain reach, state_codegen.hpp).  A centre rounded to binary32 is off by
        // <= 2^-24 B per axis, a difference of two by <= 2^-22 B per axis (its own rounding included): the FP32 distance of a
        // pair is within delta = sqrt(3) 2^-22 B of the FP64 one, and its square carries three more roundings (rho).  The
        // FP64 rule's own rounding (1e-16 relative) disappears in the slack of delta.
        double band_scale = 1.0;
        if (const char* bsc = std::getenv("STOMP_B200_SELF_BAND")) band_scale = std::max(1.0, std::atof(bsc));   // test knob: widens the undecided band
        const double B = codegen::centre_bound(r);
        const double delta = (1.7320508075688773 * std::ldexp(B, -22) * 1.05 + 1e-12) * band_scale;
        const double rho = std::ldexp(1.0, -21);
        auto down = [](double v) { float f = (float)v; if ((double)f > v) f = std::nextafterf(f, -INFINITY); return f; };
        auto up = [](double v) { float f = (float)v; if ((double)f < v) f = std::nextafterf(f, INFINITY); return f; };
        std::vector<float> lo((size_t)num_pairs), hi((size_t)num_pairs), blockf(block.size());
        for (int p = 0; p < num_pairs; ++p) {
            const double ell = r.sphere[ij[p].x].r + r.sphere[ij[p].y].r;
            const double inner = std::max(0.0, ell - delta), outer = ell + delta;
            lo[p] = down(inner * inner * (1.0 - rho));
            hi[p] = up(outer * outer * (1.0 + rho));
            e->self_structure.i.push_back(ij[p].x);
            e->self_structure.j.push_back(ij[p].y);
        }
        for (size_t b = 0; b < block.size(); ++b) {
            // bounding centres are means of up to n FP32 centres: off by a few 2^-24 B; the cull must keep every block that
            // holds a pair the bands above would not call clear
            const int na = r.sphere_begin[block[b].x + 1] - r.sphere_begin[block[b].x], nb = r.sphere_begin[block[b].y + 1] - r.sphere_begin[block[b].y];
            const double delta_b = std::ldexp(B, -17) * (1.0 + (na + nb) / 32.0);
            const double reach2 = (bound_radius[block[b].x] + bound_radius[block[b].y]) * (1.0 + 1e-6) + delta_b + 2.0 * delta;
            blockf[b] = up(reach2 * reach2 * (1.0 + 4.0 * rho));
            e->self_structure.blocks.push_back({block[b].x, block[b].y, block[b].z, block[b].w});
        }
        e->self_bands.insert(e->self_bands.end(), lo.begin(), lo.end());
        e->self_bands.insert(e->self_bands.end(), hi.begin(), hi.end());
        e->self_bands.insert(e->self_bands.end(), blockf.begin(), blockf.end());
        if (blockf.empty()) e->self_bands.push_back(0.f);
    }
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    if (e->side_stream) CUDA_TRY(e, cudaStreamSynchronize(e->side_stream));
    e->self_pairs = SelfPairs{nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0};
    for (void* p : e->self_pair_buffers) cudaFree(p);
    e->self_pair_buffers.clear();
    if (num_pairs > 0) {
        auto upload = [&](const void* src, size_t bytes, const void** dst) -> int {
            void* d = nullptr;
            CUDA_TRY(e, cudaMalloc(&d, bytes));
            e->self_pair_buffers.push_back(d);
            CUDA_TRY(e, cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
            *dst = d;
            return 0;
        };
        SelfPairs sp{nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0};
        if (int rc = upload(ij.data(), sizeof(int2) * ij.size(), (const void**)&sp.ij)) return rc;
        if (int rc = upload(limit2.data(), sizeof(double) * limit2.size(), (const void**)&sp.limit2)) return rc;
        if (int rc = upload(block.data(), sizeof(int4) * block.size(), (const void**)&sp.block)) return rc;
        if (int rc = upload(block_limit2.data(), sizeof(double) * block_limit2.size(), (const void**)&sp.block_limit2)) return rc;
        if (int rc = upload(bound.data(), sizeof(double) * bound.size(), (const void**)&sp.link_bound)) return rc;
        sp.n = num_pairs;
        sp.nblocks = (int32_t)block.size();
        e->self_pairs = sp;
    }
    return STOMP_B200_OK;
}

// (re)allocates the device grid and records its geometry; the caller fills it
static int adopt_sdf_geometry(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size)
{
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    const size_t count = (size_t)dims[0] * dims[1] * dims[2];
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    if (e->side_stream) CUDA_TRY(e, cudaStreamSynchronize(e->side_stream));
    if (e->d_sdf && e->sdf_count != count) { cudaFree(e->d_sdf); e->d_sdf = nullptr; }
    if (!e->d_sdf) {
        e->have_sdf = false;
        CUDA_TRY(e, cudaMalloc(&e->d_sdf, count * sizeof(float)));
        e->sdf_count = count;
    }
    e->sdf.grid = e->d_sdf;
    e->sdf.nx = dims[0]; e->sdf.ny = dims[1]; e->sdf.nz = dims[2];
    e->sdf.inv_h = 1.0 / voxel_size;
    e->sdf.offx = -(origin[0] * e->sdf.inv_h); e->sdf.offy = -(origin[1] * e->sdf.inv_h); e->sdf.offz = -(origin[2] * e->sdf.inv_h);
    e->sdf.wide_index = count >= ((size_t)1 << 31) ? 1 : 0;
    e->sdf_origin[0] = origin[0]; e->sdf_origin[1] = origin[1]; e->sdf_origin[2] = origin[2];
    e->sdf_voxel = voxel_size;
    e->spec_resolved = false;
    e->config_epoch++;
    return STOMP_B200_OK;
}

int stomp_b200_set_sdf(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size, const float* grid)
{
    if (!e || !dims || !origin || !grid || !(voxel_size > 0.0)) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (dims[0] < 1 || dims[1] < 1 || dims[2] < 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (int rc = adopt_sdf_geometry(e, dims, origin, voxel_size)) return rc;
    CUDA_TRY(e, cudaMemcpy(e->d_sdf, grid, e->sdf_count * sizeof(float), cudaMemcpyHostToDevice));
    e->have_sdf = true;
    return STOMP_B200_OK;
}

int stomp_b200_build_sdf_primitives(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                                    int32_t num_primitives, const int32_t* kind, const double* centre, const double* size)
{
    if (!e || !dims || !origin || !(voxel_size > 0.0) || num_primitives < 0) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (num_primitives > 0 && (!kind || !centre || !size)) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (dims[0] < 1 || dims[1] < 1 || dims[2] < 1 || dims[1] > 65535 || dims[2] > 65535) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (num_primitives > kMaxPrimitives) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "too many primitives for one call (256)");
    for (int i = 0; i < num_primitives; ++i)
        if (kind[i] < 0 || kind[i] > 2) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "primitive kind must be 0 (sphere), 1 (box) or 2 (cylinder along z)");
    if (int rc = adopt_sdf_geometry(e, dims, origin, voxel_size)) return rc;
    std::vector<PrimitiveList> host(1);
    PrimitiveList& pl = host[0];
    std::memset(&pl, 0, sizeof pl);
    pl.n = num_primitives;
    for (int i = 0; i < num_primitives; ++i) {
        pl.kind[i] = kind[i];
        for (int a = 0; a < 3; ++a) { pl.centre[i][a] = centre[3 * i + a]; pl.size[i][a] = size[3 * i + a]; }
    }
    PrimitiveList* d_list = nullptr;
    CUDA_TRY(e, cudaMalloc(&d_list, sizeof(PrimitiveList)));
    cudaError_t err = cudaMemcpy(d_list, &pl, sizeof(PrimitiveList), cudaMemcpyHostToDevice);
    if (err == cudaSuccess) {
        build_sdf_primitives_kernel<<<dim3((dims[0] + 127) / 128, dims[1], dims[2]), 128, 0, e->stream>>>(
            e->d_sdf, dims[0], dims[1], dims[2], origin[0], origin[1], origin[2], voxel_size, d_list);
        e->launch_count++;
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    cudaFree(d_list);
    if (err != cudaSuccess) { e->last_error = std::string("build_sdf_primitives: ") + cudaGetErrorString(err); return STOMP_B200_ERR_CUDA; }
    e->have_sdf = true;
    return STOMP_B200_OK;
}

// exact signed Euclidean distance transform of a device occupancy grid into e->d_sdf (geometry already adopted)
static int edt_from_device_occupancy(stomp_b200_engine* e, const uint8_t* d_occ, const char* what)
{
    const size_t count = e->sdf_count;
    const int nx = e->sdf.nx, ny = e->sdf.ny, nz = e->sdf.nz;
    int32_t* d_a = nullptr; int32_t* d_b = nullptr; int32_t* d_c = nullptr;
    auto cleanup = [&]() { cudaFree(d_a); cudaFree(d_b); cudaFree(d_c); };
    cudaError_t err = cudaMalloc(&d_a, count * sizeof(int32_t));
    if (err == cudaSuccess) err = cudaMalloc(&d_b, count * sizeof(int32_t));
    if (err == cudaSuccess) err = cudaMalloc(&d_c, count * sizeof(int32_t));
    if (err == cudaSuccess) {
        const unsigned blocks = (unsigned)((count + 255) / 256);
        edt_seed_kernel<<<blocks, 256, 0, e->stream>>>(d_occ, d_a, d_b, count);
        // three separable passes per transform: x (lines of nx, one per (y, z)), y, z; ping-pong through d_c
        auto transform = [&](int32_t* buf) {
            edt_pass_kernel<<<dim3(ny, nz), 256, sizeof(int32_t) * nx, e->stream>>>(buf, d_c, nx, 1, ny, nx, (long long)nx * ny);
            edt_pass_kernel<<<dim3(nx, nz), 256, sizeof(int32_t) * ny, e->stream>>>(d_c, buf, ny, nx, nx, 1, (long long)nx * ny);
            edt_pass_kernel<<<dim3(nx, ny), 256, sizeof(int32_t) * nz, e->stream>>>(buf, d_c, nz, (long long)nx * ny, nx, 1, nx);
            cudaMemcpyAsync(buf, d_c, count * sizeof(int32_t), cudaMemcpyDeviceToDevice, e->stream);
        };
        transform(d_a);
        transform(d_b);
        finish_edt_kernel<<<blocks, 256, 0, e->stream>>>(d_occ, d_a, d_b, e->d_sdf, e->sdf_voxel, count);
        e->launch_count += 8;
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    cleanup();
    if (err != cudaSuccess) { e->last_error = std::string(what) + ": " + cudaGetErrorString(err); return STOMP_B200_ERR_CUDA; }
    return STOMP_B200_OK;
}

int stomp_b200_build_sdf_occupancy(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                                   const uint8_t* occupied)
{
    return stomp_b200_build_sdf_scene(e, dims, origin, voxel_size, 0, nullptr, 0, 0, nullptr, nullptr, occupied);
}

int stomp_b200_build_sdf_scene(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                               int32_t num_triangles, const double* triangles, int32_t solid, int32_t num_leaves,
                               const double* leaf_centres, const double* leaf_sizes, const uint8_t* occupied)
{
    if (!e || !dims || !origin || !(voxel_size > 0.0) || num_triangles < 0 || num_leaves < 0) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if ((num_triangles > 0 && !triangles) || (num_leaves > 0 && (!leaf_centres || !leaf_sizes))) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (dims[0] < 1 || dims[1] < 1 || dims[2] < 1 || dims[0] > 1024 || dims[1] > 1024 || dims[2] > 1024)
        return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "occupancy grids are limited to 1024 voxels per axis (exact int32 squared distances)");
    for (size_t i = 0; i < (size_t)num_triangles * 9; ++i)
        if (!(std::fabs(triangles[i]) <= 1e9)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "mesh vertex is not finite");
    for (int i = 0; i < num_leaves; ++i)
        if (!(leaf_sizes[i] > 0.0) || !(std::fabs(leaf_centres[3 * i]) <= 1e9) || !(std::fabs(leaf_centres[3 * i + 1]) <= 1e9) || !(std::fabs(leaf_centres[3 * i + 2]) <= 1e9))
            return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "octomap leaf: centre not finite or size not positive");
    if (int rc = adopt_sdf_geometry(e, dims, origin, voxel_size)) return rc;
    const size_t count = e->sdf_count;
    const int nx = dims[0], ny = dims[1], nz = dims[2];
    uint8_t* d_occ = nullptr; uint8_t* d_out = nullptr; double* d_tri = nullptr; double* d_leaf = nullptr; int* d_flag = nullptr;
    auto cleanup = [&]() { cudaFree(d_occ); cudaFree(d_out); cudaFree(d_tri); cudaFree(d_leaf); cudaFree(d_flag); };
    cudaError_t err = cudaMalloc(&d_occ, count);
    if (err == cudaSuccess) err = occupied ? cudaMemcpyAsync(d_occ, occupied, count, cudaMemcpyHostToDevice, e->stream) : cudaMemsetAsync(d_occ, 0, count, e->stream);
    if (err == cudaSuccess && num_triangles > 0) {
        err = cudaMalloc(&d_tri, sizeof(double) * 9 * (size_t)num_triangles);
        if (err == cudaSuccess) err = cudaMemcpyAsync(d_tri, triangles, sizeof(double) * 9 * (size_t)num_triangles, cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) {
            voxelise_triangles_kernel<<<num_triangles, 128, 0, e->stream>>>(d_tri, num_triangles, d_occ, nx, ny, nz, origin[0], origin[1], origin[2], voxel_size);
            e->launch_count++;
            err = cudaGetLastError();
        }
        if (err == cudaSuccess && solid) {      // interior of the closed shells: free voxels the boundary cannot reach
            err = cudaMalloc(&d_out, count);
            if (err == cudaSuccess) err = cudaMalloc(&d_flag, sizeof(int));
            if (err == cudaSuccess) {
                flood_seed_kernel<<<(unsigned)((count + 255) / 256), 256, 0, e->stream>>>(d_occ, d_out, nx, ny, nz);
                e->launch_count++;
                for (int round = 0; round < 4096 && err == cudaSuccess; ++round) {
                    int changed = 0;
                    err = cudaMemsetAsync(d_flag, 0, sizeof(int), e->stream);
                    flood_sweep_kernel<<<(ny * nz + 127) / 128, 128, 0, e->stream>>>(d_occ, d_out, nx, 1, ny, nx, nz, (long long)nx * ny, d_flag);
                    flood_sweep_kernel<<<(nx * nz + 127) / 128, 128, 0, e->stream>>>(d_occ, d_out, ny, nx, nx, 1, nz, (long long)nx * ny, d_flag);
                    flood_sweep_kernel<<<(nx * ny + 127) / 128, 128, 0, e->stream>>>(d_occ, d_out, nz, (long long)nx * ny, nx, 1, ny, nx, d_flag);
                    e->launch_count += 3;
                    if (err == cudaSuccess) err = cudaMemcpyAsync(&changed, d_flag, sizeof(int), cudaMemcpyDeviceToHost, e->stream);
                    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
                    if (!changed) break;
                }
                if (err == cudaSuccess) {
                    flood_fill_kernel<<<(unsigned)((count + 255) / 256), 256, 0, e->stream>>>(d_occ, d_out, count);
                    e->launch_count++;
                    err = cudaGetLastError();
                }
            }
        }
    }
    if (err == cudaSuccess && num_leaves > 0) {
        err = cudaMalloc(&d_leaf, sizeof(double) * 4 * (size_t)num_leaves);
        if (err == cudaSuccess) err = cudaMemcpyAsync(d_leaf, leaf_centres, sizeof(double) * 3 * (size_t)num_leaves, cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) err = cudaMemcpyAsync(d_leaf + 3 * (size_t)num_leaves, leaf_sizes, sizeof(double) * (size_t)num_leaves, cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) {
            voxelise_leaves_kernel<<<num_leaves, 32, 0, e->stream>>>(d_leaf, d_leaf + 3 * (size_t)num_leaves, num_leaves, d_occ, nx, ny, nz, origin[0], origin[1], origin[2], voxel_size);
            e->launch_count++;
            err = cudaGetLastError();
        }
    }
    if (err != cudaSuccess) { cleanup(); e->last_error = std::string("build_sdf_scene: ") + cudaGetErrorString(err); return STOMP_B200_ERR_CUDA; }
    const int rc = edt_from_device_occupancy(e, d_occ, "build_sdf_scene");
    cleanup();
    if (rc) return rc;
    e->have_sdf = true;
    return STOMP_B200_OK;
}

int stomp_b200_get_sdf(stomp_b200_engine* e, float* out, size_t count, int32_t dims_out[3], double origin_out[3], double* voxel_size_out)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_sdf) return fail(e, STOMP_B200_ERR_NOT_READY, "no distance field set");
    if (dims_out) { dims_out[0] = e->sdf.nx; dims_out[1] = e->sdf.ny; dims_out[2] = e->sdf.nz; }
    if (origin_out) { origin_out[0] = e->sdf_origin[0]; origin_out[1] = e->sdf_origin[1]; origin_out[2] = e->sdf_origin[2]; }
    if (voxel_size_out) *voxel_size_out = e->sdf_voxel;
    if (out) {
        if (count != e->sdf_count) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "count does not match the grid");
        CUDA_TRY(e, cudaSetDevice(e->cfg.device));
        CUDA_TRY(e, cudaStreamSynchronize(e->stream));
        CUDA_TRY(e, cudaMemcpy(out, e->d_sdf, count * sizeof(float), cudaMemcpyDeviceToHost));
    }
    return STOMP_B200_OK;
}

// Rows of B = L^-1 for the recurrence sampler (kernels.cuh: sample_rollouts_banded_kernel).  R = U U^T with U upper
// triangular and banded (Cholesky run from the last row up, long double), B = U^T.  The table is accepted only if the
// recurrence reproduces columns of the caller's L (so a caller that hands in some other factor keeps the contraction).
static bool build_sampler_band(const double* R, const double* L, int T, int hw, std::vector<double>& table)
{
    if (hw < 1 || hw > kRBand) return false;
    std::vector<long double> U((size_t)T * (hw + 1), 0.0L);      // U[i][i + o] at [i][o]
    auto u = [&](int i, int k) -> long double& { return U[(size_t)i * (hw + 1) + (k - i)]; };
    for (int j = T - 1; j >= 0; --j) {
        long double sdiag = R[(size_t)j * T + j];
        for (int k = j + 1; k <= std::min(T - 1, j + hw); ++k) sdiag -= u(j, k) * u(j, k);
        if (!(sdiag > 0.0L)) return false;
        u(j, j) = sqrtl(sdiag);
        for (int i = j - 1; i >= std::max(0, j - hw); --i) {
            long double sij = R[(size_t)i * T + j];
            for (int k = j + 1; k <= std::min(T - 1, i + hw); ++k) sij -= u(i, k) * u(j, k);
            u(i, j) = sij / u(j, j);
        }
    }
    table.assign((size_t)T * 8, 0.0);
    for (int t = 0; t < T; ++t) {
        const long double inv = 1.0L / u(t, t);
        table[(size_t)t * 8] = (double)inv;
        for (int o = 1; o <= hw && t - o >= 0; ++o) table[(size_t)t * 8 + o] = (double)(u(t - o, t) * inv);
    }
    // check against the given L: the recurrence applied to unit vectors must give columns of L
    double lmax = 0.0;
    for (size_t i = 0; i < (size_t)T * T; ++i) lmax = std::max(lmax, std::fabs(L[i]));
    const int cols[3] = {0, T / 3, T - 1};
    std::vector<double> n(T);
    for (int c : cols) {
        for (int t = 0; t < T; ++t) {
            double acc = (t == c ? 1.0 : 0.0) * table[(size_t)t * 8];
            for (int o = 1; o <= hw && t - o >= 0; ++o) acc -= table[(size_t)t * 8 + o] * n[t - o];
            n[t] = acc;
            if (!(std::fabs(n[t] - L[(size_t)t * T + c]) <= 1e-6 * lmax)) return false;
        }
    }
    return true;
}

int stomp_b200_set_control_cost_matrices(stomp_b200_engine* e, const double* R, const double* Rinv, const double* L)
{
    if (!e || !R || !L) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    const int T = e->T;
    if (e->cfg.use_projection) {
        // PolicyImprovement::preComputeProjectionMatrices (PolicyImprovement.cpp:750-801): M = R^-1 with column p scaled by
        // 1 / (T * R^-1[p][p]); its inverse by LU with complete pivoting, as Eigen's fullPivLu().inverse() (:795)
        if (!Rinv) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "use_projection needs Rinv");
        host::Dense M(T, T), Minv;
        for (int pcol = 0; pcol < T; ++pcol) {
            const double column_max = Rinv[(size_t)pcol * T + pcol];
            const double f = 1.0 / (T * column_max);
            for (int i = 0; i < T; ++i) M.at(i, pcol) = Rinv[(size_t)i * T + pcol] * f;
        }
        if (!host::invert_full_pivot(M, Minv)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "the projection matrix is singular");
        CUDA_TRY(e, cudaStreamSynchronize(e->stream));
        CUDA_TRY(e, cudaMemcpy(e->d_Mproj, M.data(), sizeof(double) * T * T, cudaMemcpyHostToDevice));
        CUDA_TRY(e, cudaMemcpy(e->d_Minv, Minv.data(), sizeof(double) * T * T, cudaMemcpyHostToDevice));
        e->base.Mproj = e->d_Mproj;
        e->base.Minv = e->d_Minv;
    }
    std::vector<double> Lt((size_t)T * T), band((size_t)T * (2 * kRBand + 1), 0.0);
    for (int t = 0; t < T; ++t)
        for (int u = 0; u < T; ++u) {
            Lt[(size_t)u * T + t] = (u <= t) ? L[(size_t)t * T + u] : 0.0;
            const int o = u - t + kRBand;
            if (o >= 0 && o <= 2 * kRBand) band[(size_t)t * (2 * kRBand + 1) + o] = R[(size_t)t * T + u];
            else if (R[(size_t)t * T + u] != 0.0)
                return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "R has entries outside the 13-wide band of 7-tap rules");
        }
    int hw = 0;
    for (int t = 0; t < T; ++t)
        for (int o = 1; o <= kRBand; ++o)
            if (band[(size_t)t * (2 * kRBand + 1) + kRBand + o] != 0.0) hw = std::max(hw, o);
    e->base.rband_halfwidth = hw;
    // R built from the 7-tap rules is Toeplitz inside its band (DESIGN.md): keep the diagonals as kernel parameters
    e->base.r_toeplitz = 1;
    for (int o = 0; o <= kRBand; ++o) e->base.r_diag[o] = band[kRBand + o];
    for (int t = 0; t < T && e->base.r_toeplitz; ++t)
        for (int o = 0; o <= kRBand && t + o < T; ++o)
            if (band[(size_t)t * (2 * kRBand + 1) + kRBand + o] != e->base.r_diag[o]) { e->base.r_toeplitz = 0; break; }
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    {
        std::vector<double> table;
        if (build_sampler_band(R, L, T, hw, table)) {
            CUDA_TRY(e, cudaMemcpy(e->d_Lband, table.data(), sizeof(double) * table.size(), cudaMemcpyHostToDevice));
            e->base.Lband = e->d_Lband;
            e->base.lband_halfwidth = hw;
        } else {
            e->base.Lband = nullptr;
            e->base.lband_halfwidth = 0;
        }
    }
    CUDA_TRY(e, cudaMemcpy(const_cast<double*>(e->base.Lt), Lt.data(), sizeof(double) * Lt.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(e, cudaMemcpy(const_cast<double*>(e->base.Rband), band.data(), sizeof(double) * band.size(), cudaMemcpyHostToDevice));
    e->have_matrices = true;
    e->config_epoch++;
    return STOMP_B200_OK;
}

int stomp_b200_set_policies(stomp_b200_engine* e, int32_t first_query, int32_t count, const double* parameters_all, const double* min_control_cost)
{
    if (!e || !parameters_all || !min_control_cost) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (count < 1 || first_query < 0 || first_query + count > e->Q) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "query range out of bounds");
    const size_t na = (size_t)e->D * e->N, nm = (size_t)e->D * e->T;
    // NaN / infinite / absurd joint values never reach the kernels (the reference rejects NaN in checkNaN,
    // src/MotionPlanners.cpp:563-571); 1e6 rad or m is far beyond any joint and far below where the deterministic
    // sin / cos reduction stops being exact
    for (size_t i = 0; i < na * count; ++i)
        if (!(std::fabs(parameters_all[i]) <= 1e6)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "parameters_all holds a NaN, an infinity or a value beyond 1e6");
    for (size_t i = 0; i < nm * count; ++i)
        if (!(std::fabs(min_control_cost[i]) <= 1e6)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "min_control_cost holds a NaN, an infinity or a value beyond 1e6");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;      // an owed noise-less rollout belongs to the policy as it is now
    e->scalars_fresh = false; e->solution_fresh = false;
    // stream-ordered copies out of pinned staging (theta rows of all queries, then the min-control-cost rows: the two device
    // tensors are query-major too, so a batch is two copies): no synchronisation, the caller's buffers are free on return
    const size_t total = (na + nm) * (size_t)e->Q;
    if (!e->h_policy && sizeof(double) * total <= ((size_t)256 << 20))
        if (cudaMallocHost(&e->h_policy, sizeof(double) * total) != cudaSuccess) { e->h_policy = nullptr; cudaGetLastError(); }
    double* d_theta = e->base.theta_all + (size_t)first_query * na;
    double* d_mincc = const_cast<double*>(e->base.mincc) + (size_t)first_query * nm;
    if (e->h_policy) {
        bool busy = false;
        for (int q = first_query; q < first_query + count; ++q) busy = busy || e->policy_in_flight[q];
        if (busy) {      // a slot's previous copy may still be reading it
            CUDA_TRY(e, cudaEventSynchronize(e->ev_policy));
            std::fill(e->policy_in_flight.begin(), e->policy_in_flight.end(), 0);
        }
        double* stage_theta = e->h_policy + (size_t)first_query * na;
        double* stage_mincc = e->h_policy + (size_t)e->Q * na + (size_t)first_query * nm;
        std::memcpy(stage_theta, parameters_all, sizeof(double) * na * count);
        std::memcpy(stage_mincc, min_control_cost, sizeof(double) * nm * count);
        CUDA_TRY(e, cudaMemcpyAsync(d_theta, stage_theta, sizeof(double) * na * count, cudaMemcpyHostToDevice, e->stream));
        CUDA_TRY(e, cudaMemcpyAsync(d_mincc, stage_mincc, sizeof(double) * nm * count, cudaMemcpyHostToDevice, e->stream));
        CUDA_TRY(e, cudaEventRecord(e->ev_policy, e->stream));
        for (int q = first_query; q < first_query + count; ++q) e->policy_in_flight[q] = 1;
    } else {
        CUDA_TRY(e, cudaStreamSynchronize(e->stream));
        CUDA_TRY(e, cudaMemcpy(d_theta, parameters_all, sizeof(double) * na * count, cudaMemcpyHostToDevice));
        CUDA_TRY(e, cudaMemcpy(d_mincc, min_control_cost, sizeof(double) * nm * count, cudaMemcpyHostToDevice));
    }
    for (int q = first_query; q < first_query + count; ++q) e->have_policy[q] = 1;
    e->loop.edge_dirty = true;
    return STOMP_B200_OK;
}

int stomp_b200_set_policy(stomp_b200_engine* e, int32_t query, const double* parameters_all, const double* min_control_cost)
{
    return stomp_b200_set_policies(e, query, 1, parameters_all, min_control_cost);
}

int stomp_b200_host_policy(int32_t num_time_steps, int32_t num_dimensions, double movement_duration,
                           const double derivative_weights[4], const double* initial_all, int32_t set_to_min_control_cost,
                           double* R, double* Rinv, double* L, double* parameters_all_out, double* min_control_cost_out)
{
    if (!derivative_weights || !initial_all || num_time_steps < 2 || num_dimensions < 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    host::PolicyCore pc;
    if (!pc.initialize(num_time_steps, num_dimensions, movement_duration, derivative_weights, initial_all))
        return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (set_to_min_control_cost) pc.setToMinControlCost();
    else pc.updateMinControlCostParameters(pc.params_all.data());
    const size_t T = num_time_steps;
    if (R) std::memcpy(R, pc.R.data(), sizeof(double) * T * T);
    if (Rinv) std::memcpy(Rinv, pc.Rinv.data(), sizeof(double) * T * T);
    if (L) std::memcpy(L, pc.L.data(), sizeof(double) * T * T);
    if (parameters_all_out) std::memcpy(parameters_all_out, pc.params_all.data(), sizeof(double) * pc.params_all.size());
    if (min_control_cost_out) std::memcpy(min_control_cost_out, pc.mincc.data(), sizeof(double) * pc.mincc.size());
    return STOMP_B200_OK;
}

int stomp_b200_host_initial_trajectory(int32_t num_time_steps, int32_t num_dimensions, const double* start,
                                       const double* goal, double* initial_all)
{
    if (!start || !goal || !initial_all || num_time_steps < 2 || num_dimensions < 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    host::linear_initial_trajectory(num_time_steps, num_dimensions, start, goal, initial_all);
    return STOMP_B200_OK;
}

int stomp_b200_begin_solve(stomp_b200_engine* e)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (int rc = ready_to_solve(e)) return rc;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    e->loop.num_rollouts = 0;
    e->loop.noiseless_valid = false;
    e->loop.adapted_valid = false;
    e->loop.last_gen = 0; e->loop.last_local = 0; e->loop.last_noiseless_slot = -1;
    if (int rc = join_side_stream(e)) return rc;
    e->loop.nl_deferred = false;
    e->scalars_fresh = false; e->solution_fresh = false;
    if (e->h_note) {
        // the progress words are reset from the host: no kernel that could still write them may be in flight (after a
        // finish_solve none is; policy uploads queued since are copies)
        if (e->note_writers_in_flight) {
            CUDA_TRY(e, cudaStreamSynchronize(e->stream));
            e->note_writers_in_flight = false;
        }
        for (int i = 0; i < 2 * e->Q; ++i) e->h_note[i] = 0;
    }
    CUDA_TRY(e, cudaMemsetAsync(e->d_nl_counter, 0, sizeof(uint32_t) * e->Q, e->stream));
    reset_solve_state_kernel<<<(e->Q + 127) / 128, 128, 0, e->stream>>>(e->base);
    e->launch_count++;
    if (int rc = check_launch(e, "reset_solve_state_kernel")) return rc;
    e->loop.edge_dirty = true;
    e->solving = true;
    return STOMP_B200_OK;
}

int32_t stomp_b200_next_num_generated(const stomp_b200_engine* e)
{
    if (!e) return 0;
    return plan_rollouts(e).gen_local;
}

int stomp_b200_iterate(stomp_b200_engine* e, int32_t iteration, const double* unit_noise, const double* epsilon,
                       double* noiseless_total_cost, uint8_t* noiseless_valid, int32_t* stop)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->solving) return fail(e, STOMP_B200_ERR_NOT_READY, "stomp_b200_begin_solve first");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    const size_t count = (size_t)e->Q * stomp_b200_next_num_generated(e) * e->D * e->T;
    int mode = kNoisePhilox;
    if (unit_noise) {
        mode = kNoiseUnit;
        CUDA_TRY(e, cudaMemcpyAsync(e->base.unit_noise, unit_noise, sizeof(double) * count, cudaMemcpyHostToDevice, e->stream));
    } else if (epsilon) {
        mode = kNoiseEpsilon;
        CUDA_TRY(e, cudaMemcpyAsync(e->base.epsilon, epsilon, sizeof(double) * count, cudaMemcpyHostToDevice, e->stream));
    }
    if (int rc = iterate_async(e, iteration, mode, 0)) return rc;
    if (int rc = fetch_query_scalars(e)) return rc;
    for (int q = 0; q < e->Q; ++q) {
        if (noiseless_total_cost) noiseless_total_cost[q] = e->h_cost[q];
        if (noiseless_valid) noiseless_valid[q] = e->h_valid[q];
        if (stop) stop[q] = e->h_stop[q];
    }
    return STOMP_B200_OK;
}

int stomp_b200_run(stomp_b200_engine* e, int32_t first_iteration, int32_t num_iterations, int32_t honour_stop)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->solving) return fail(e, STOMP_B200_ERR_NOT_READY, "stomp_b200_begin_solve first");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    // a lone iteration whose end the caller waits for: three plain launches start sooner than one graph launch (an isolated
    // C3 iteration: 88 us against 97 us); queued back to back the graph wins (57 against 61 us per iteration)
    const bool allow_graph = num_iterations > 1;
    // the first call inside a timed region starts it: the stream is idle since stomp_b200_timer_begin, and what lies between
    // that call and this one is the caller's own time (the interpreter of bench.py), not a step's
    if (e->timer_armed && !e->timer_end_recorded) CUDA_TRY(e, cudaEventRecord(e->timer_a, e->stream));
    for (int i = 0; i < num_iterations; ++i)
        if (int rc = iterate_async(e, first_iteration + i, kNoisePhilox, honour_stop ? 1 : 0, allow_graph)) return rc;
    if (int rc = join_side_stream(e)) return rc;
    // a timed region (stomp_b200_timer_begin) ends where the device finishes the last kernel queued above: the end event goes
    // in before the host waits, so that the bracket holds device work and launch latency but not the host's wake-up from the
    // wait and its way back to stomp_b200_timer_end (5 - 10 us, an eighth of an isolated C3 iteration)
    if (e->timer_armed) { CUDA_TRY(e, cudaEventRecord(e->timer_b, e->stream)); e->timer_end_recorded = true; }
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    e->note_writers_in_flight = false;
    resolve_profile(e);
    return STOMP_B200_OK;
}

int stomp_b200_solve(stomp_b200_engine* e, int32_t max_iterations, int32_t poll_every, int32_t* iterations_run)
{
    if (!e || max_iterations < 0) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->solving) return fail(e, STOMP_B200_ERR_NOT_READY, "stomp_b200_begin_solve first");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (poll_every <= 0) poll_every = 8;
    int done = 0;
    // Paced by the device's progress words (one query set on one GPU, or query sharding: no exchange couples the ranks):
    // iteration i is queued once the noise-less rollout of iteration i - 1 - solve_ahead has been recorded, so the device
    // never runs dry (the rest of the running iteration is the host's slack) and at most solve_ahead iterations are queued
    // behind a stop.  One synchronisation per call, at the end.  Rollout sharding keeps the synchronising poll loop: every
    // rank has to queue the same iterations (the exchange epochs are counted per queued iteration).
    const bool paced = e->h_note != nullptr && e->solve_ahead > 0 && !(e->cfg.shard_mode == 0 && e->cfg.world_size > 1);
    if (paced) {
        unsigned spins = 0;
        while (done < max_iterations) {
            bool all_stopped = true;
            int recorded = INT32_MAX;
            for (int q = 0; q < e->Q; ++q) {
                if (e->h_note[2 * q + 1] != 0) continue;
                all_stopped = false;
                { const int r = e->h_note[2 * q]; if (r < recorded) recorded = r; }
            }
            if (all_stopped) break;
            bool go = done <= recorded + e->solve_ahead;
            if (!go && (++spins & 255u) == 0) {
                // nothing left on the stream and still no word: the record rides on a launch that is not queued yet
                const cudaError_t qs = cudaStreamQuery(e->stream);
                if (qs == cudaSuccess) go = true;
                else if (qs != cudaErrorNotReady) { e->last_error = std::string("stomp_b200_solve: ") + cudaGetErrorString(qs); return STOMP_B200_ERR_CUDA; }
            }
            if (!go) {
#if defined(__x86_64__) || defined(__i386__)
                __builtin_ia32_pause();
#endif
                continue;
            }
            if (int rc = iterate_async(e, done, kNoisePhilox, 1)) return rc;
            ++done;
            spins = 0;
        }
        if (int rc = fetch_query_scalars(e, true)) return rc;
        if (iterations_run) *iterations_run = done;
        return STOMP_B200_OK;
    }
    while (done < max_iterations) {
        const int n = std::min(poll_every, max_iterations - done);
        for (int i = 0; i < n; ++i)
            if (int rc = iterate_async(e, done + i, kNoisePhilox, 1)) return rc;
        done += n;
        // one pinned block, one synchronisation per poll; a small solution rides along so that finish_solve finds it there
        const bool small_solution = sizeof(double) * (size_t)e->Q * e->D * e->T <= ((size_t)256 << 10);
        if (int rc = fetch_query_scalars(e, small_solution)) return rc;
        bool all_stopped = true;
        for (int q = 0; q < e->Q && all_stopped; ++q) all_stopped = e->h_stop[q] != 0;
        if (all_stopped) break;
    }
    if (iterations_run) *iterations_run = done;
    return STOMP_B200_OK;
}

int stomp_b200_finish_solve(stomp_b200_engine* e, double* solution, int32_t* status, int32_t* iterations_used,
                            double* noiseless_total_cost)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    // straight after stomp_b200_solve both mirrors are current and no device call is made here
    if (!e->scalars_fresh || (solution && !e->solution_fresh))
        if (int rc = fetch_query_scalars(e, solution != nullptr)) return rc;
    if (solution) {
        // parameters_all_[d][6 + t]  (StompPlanner.cpp:148-163)
        if (e->solution_fresh) std::memcpy(solution, e->h_solution, sizeof(double) * (size_t)e->Q * e->D * e->T);
        else CUDA_TRY(e, cudaMemcpy2D(solution, sizeof(double) * e->T, e->base.theta_all + kPad, sizeof(double) * e->N,
                                      sizeof(double) * e->T, (size_t)e->Q * e->D, cudaMemcpyDeviceToHost));
    }
    for (int q = 0; q < e->Q; ++q) {
        if (status)
            status[q] = ((e->h_cost[q] < 1) && (std::fabs(e->h_impr[q]) <= e->cfg.min_cost_improvement)) ? 1 : 0;
        if (iterations_used) iterations_used[q] = e->h_iters[q];
        if (noiseless_total_cost) noiseless_total_cost[q] = e->h_cost[q];
    }
    e->solving = false;
    return STOMP_B200_OK;
}

int stomp_b200_num_rollouts(const stomp_b200_engine* e, int32_t* num_rollouts, int32_t* num_generated)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (num_rollouts) *num_rollouts = e->loop.num_rollouts;
    if (num_generated) *num_generated = e->loop.last_gen;
    return STOMP_B200_OK;
}

int stomp_b200_get_tensor(stomp_b200_engine* e, int32_t tensor, void* out, size_t out_bytes)
{
    if (!e || !out) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    const LoopParams& b = e->base;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    resolve_profile(e);
    if (tensor == STOMP_B200_CUMULATIVE_COSTS || tensor == STOMP_B200_FULL_COSTS || tensor == STOMP_B200_TOTAL_COST ||
        tensor == STOMP_B200_PROBABILITIES || tensor == STOMP_B200_FULL_PROBABILITIES)
        if (int rc = gather_tables_for_readback(e)) return rc;
    const size_t Q = e->Q, T = e->T, D = e->D, N = e->N;
    const size_t nl = e->loop.last_local;     // local rollouts of the last iteration
    const size_t ng = e->loop.num_rollouts;   // rollouts in the rollout-indexed tables
    // copy `rows` rows of `row_bytes` per query out of a [Q][stride_rows] table
    auto per_query = [&](const void* src, size_t rows, size_t stride_rows, size_t row_bytes) -> int {
        if (out_bytes != Q * rows * row_bytes) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
        if (rows == 0) return 0;
        CUDA_TRY(e, cudaMemcpy2D(out, rows * row_bytes, src, stride_rows * row_bytes, rows * row_bytes, Q, cudaMemcpyDeviceToHost));
        return 0;
    };
    auto from_sums = [&](int kind) -> int {   // 5 cumulative, 6 full, 7 total
        const size_t width = kind == 7 ? 1 : D;
        if (out_bytes != Q * ng * width * sizeof(double)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
        std::vector<double> s(Q * e->gslots * e->sumw);
        CUDA_TRY(e, cudaMemcpy(s.data(), b.sums, sizeof(double) * s.size(), cudaMemcpyDeviceToHost));
        double* o = static_cast<double*>(out);
        for (size_t q = 0; q < Q; ++q)
            for (size_t k = 0; k < ng; ++k) {
                const double* r = s.data() + (q * e->gslots + k) * e->sumw;
                if (kind == 7) {
                    double c = r[0];
                    for (size_t d = 0; d < D; ++d) c += r[1 + d];
                    o[q * ng + k] = c;
                } else {
                    for (size_t d = 0; d < D; ++d) o[(q * ng + k) * D + d] = r[0] + r[1 + d];   // cumulative (= sum_t state + control_d) and full costs
                }
            }
        return 0;
    };
    switch (tensor) {
        case STOMP_B200_ROLLOUTS: return per_query(b.rollouts, nl * D, (size_t)e->slots * D, T * sizeof(double));
        case STOMP_B200_NOISE:
            if (e->loop.last_noise_from_rollouts) return fail(e, STOMP_B200_ERR_NOT_READY, "noise_ was not materialised in this configuration (keep_debug_tensors keeps it)");
            return per_query(b.noise, nl * D, (size_t)e->slots * D, T * sizeof(double));
        case STOMP_B200_STATE_COSTS: return per_query(b.state_costs, nl, e->slots, T * sizeof(double));
        case STOMP_B200_VERDICTS: return per_query(b.verdicts, nl, e->slots, T);
        case STOMP_B200_CONTROL_COSTS:
            if (!b.control_costs) return fail(e, STOMP_B200_ERR_NOT_READY, "control costs need keep_debug_tensors");
            return per_query(b.control_costs, nl * D, (size_t)e->slots * D, T * sizeof(double));
        case STOMP_B200_CUMULATIVE_COSTS:
            if (e->cfg.use_cumulative_costs != 1) return fail(e, STOMP_B200_ERR_UNSUPPORTED, "per-time-step / forward-cumulation mode: cumulative costs follow from state costs + control costs, read those");
            return from_sums(5);
        case STOMP_B200_FULL_COSTS: return from_sums(6);
        case STOMP_B200_TOTAL_COST: return from_sums(7);
        case STOMP_B200_PROBABILITIES:
            if (e->cfg.use_cumulative_costs != 1) return per_query(b.pt_prob, ng * D, (size_t)e->gslots * D, T * sizeof(double));
            // fall through
        case STOMP_B200_FULL_PROBABILITIES: {
            // the device tables hold exp(-h (c - min) / den); divide by their sum (wpart), exactly as
            // weighted_update_kernel does (probabilities_ and full_probabilities_ coincide here)
            const size_t width = tensor == STOMP_B200_PROBABILITIES ? T : 1;
            if (out_bytes != Q * ng * D * width * sizeof(double)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
            std::vector<double> pr(Q * e->gslots * D), part(Q * D * b.wblocks_cap);
            CUDA_TRY(e, cudaMemcpy(pr.data(), b.prob, sizeof(double) * pr.size(), cudaMemcpyDeviceToHost));
            CUDA_TRY(e, cudaMemcpy(part.data(), b.wpart, sizeof(double) * part.size(), cudaMemcpyDeviceToHost));
            const int wblocks = e->loop.last_wblocks;   // as launched
            double* o = static_cast<double*>(out);
            for (size_t q = 0; q < Q; ++q)
                for (size_t d = 0; d < D; ++d) {
                    double psum = 0.0;
                    for (int bl = 0; bl < wblocks; ++bl) psum += part[(q * D + d) * b.wblocks_cap + bl];
                    for (size_t k = 0; k < ng; ++k) {
                        const double v = pr[(q * e->gslots + k) * D + d] / psum;
                        for (size_t t = 0; t < width; ++t) o[((q * ng + k) * D + d) * width + t] = v;
                    }
                }
            return 0;
        }
        case STOMP_B200_UPDATES: return per_query(b.updates, 1, 1, D * T * sizeof(double));
        case STOMP_B200_PARAMETERS:
            if (out_bytes != Q * D * T * sizeof(double)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
            CUDA_TRY(e, cudaMemcpy2D(out, sizeof(double) * T, b.theta_all + kPad, sizeof(double) * N, sizeof(double) * T, Q * D, cudaMemcpyDeviceToHost));
            return 0;
        case STOMP_B200_PARAMETERS_ALL: return per_query(b.theta_all, 1, 1, D * N * sizeof(double));
        case STOMP_B200_STDDEVS: return per_query(b.sigma, 1, 1, D * sizeof(double));
        case STOMP_B200_NOISELESS_STATE_COSTS: return per_query(b.nl_state, 1, 1, T * sizeof(double));
        case STOMP_B200_NOISELESS_CONTROL_COSTS: return per_query(b.nl_control, 1, 1, D * T * sizeof(double));
        case STOMP_B200_UNIT_NOISE: {
            const size_t cap = (size_t)std::max(e->cfg.num_rollouts_per_iteration, e->cfg.min_rollouts) / (e->cfg.shard_mode == 0 ? e->cfg.world_size : 1) + 1;
            (void)cap;
            // staging layout is [Q][G][D][T] with G = rollouts generated in the last iteration (dense)
            if (out_bytes != Q * e->loop.last_gen * D * T * sizeof(double)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
            CUDA_TRY(e, cudaMemcpy(out, b.unit_noise, out_bytes, cudaMemcpyDeviceToHost));
            return 0;
        }
        case STOMP_B200_EPSILON:
            if (out_bytes != Q * e->loop.last_gen * D * T * sizeof(double)) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "out_bytes does not match the tensor size");
            CUDA_TRY(e, cudaMemcpy(out, b.epsilon, out_bytes, cudaMemcpyDeviceToHost));
            return 0;
        case STOMP_B200_ROLLOUT_VALIDITY: return per_query(b.validity, e->loop.last_gen, e->slots, 1);
        case STOMP_B200_NOISE_PROJECTED:
            if (!b.noise_proj) return fail(e, STOMP_B200_ERR_NOT_READY, "noise_projected_ exists with use_projection only (it is noise_ otherwise)");
            return per_query(b.noise_proj, nl * D, (size_t)e->slots * D, T * sizeof(double));
        case STOMP_B200_ROLLOUTS_PROJECTED:
            if (!b.proj) return fail(e, STOMP_B200_ERR_NOT_READY, "parameters_noise_projected_ is kept in configurations with rollout reuse only");
            return per_query(b.proj, nl * D, (size_t)e->slots * D, T * sizeof(double));
        default: return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "unknown tensor id");
    }
}

// grow-only device scratch of stomp_b200_evaluate_states (the start / goal validity path calls it per query)
static int eval_scratch(stomp_b200_engine* e, size_t states, size_t trajectories)
{
    if (states * e->D > e->eval_cap_theta) {
        if (e->eval_theta) cudaFree(e->eval_theta);
        e->eval_theta = nullptr; e->eval_cap_theta = 0;
        const size_t cap = std::max<size_t>(states * e->D, 1024);
        CUDA_TRY(e, cudaMalloc(&e->eval_theta, sizeof(double) * cap));
        e->eval_cap_theta = cap;
    }
    if (states > e->eval_cap_states) {
        if (e->eval_cost) cudaFree(e->eval_cost);
        if (e->eval_verdict) cudaFree(e->eval_verdict);
        e->eval_cost = nullptr; e->eval_verdict = nullptr; e->eval_cap_states = 0;
        const size_t cap = std::max<size_t>(states, 1024);
        CUDA_TRY(e, cudaMalloc(&e->eval_cost, sizeof(double) * cap));
        CUDA_TRY(e, cudaMalloc(&e->eval_verdict, cap));
        e->eval_cap_states = cap;
    }
    if (trajectories > e->eval_cap_traj) {
        if (e->eval_valid) cudaFree(e->eval_valid);
        e->eval_valid = nullptr; e->eval_cap_traj = 0;
        const size_t cap = std::max<size_t>(trajectories, 256);
        CUDA_TRY(e, cudaMalloc(&e->eval_valid, cap));
        e->eval_cap_traj = cap;
    }
    return 0;
}

int stomp_b200_evaluate_states(stomp_b200_engine* e, const double* theta, int32_t num_trajectories, int32_t num_steps,
                               double* state_costs, uint8_t* verdicts, uint8_t* validity)
{
    if (!e || !theta || num_trajectories < 1 || num_steps < 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_chain || !e->have_spheres || !e->have_sdf) return fail(e, STOMP_B200_ERR_NOT_READY, "chain, spheres and SDF must be set first");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    const size_t states = (size_t)num_trajectories * num_steps;
    if (states > (size_t)0x7fffff00) return fail(e, STOMP_B200_ERR_INVALID_ARGUMENT, "too many states for one call");
    if (int rc = eval_scratch(e, states, (size_t)num_trajectories)) return rc;
    double* d_theta = e->eval_theta; double* d_cost = e->eval_cost; uint8_t* d_verdict = e->eval_verdict; uint8_t* d_valid = e->eval_valid;
    // the run-time specialised kernel drops index clamps it can prove redundant for sane joint values; values it cannot
    // vouch for (NaN, infinities, |q| > 1e6) go through the generic kernel, which clamps and converts with saturation
    bool sane = true;
    for (size_t i = 0; i < states * e->D && sane; ++i) sane = std::fabs(theta[i]) <= 1e6;
    CUDA_TRY(e, cudaMemcpyAsync(d_theta, theta, sizeof(double) * states * e->D, cudaMemcpyHostToDevice, e->stream));
    {
        Scope sc(e, STOMP_B200_KERNEL_COST);
        const StateKernelArgs a = trajectory_state_args(e, d_theta, num_trajectories, num_steps, d_cost, d_verdict, d_valid);
        if (int rc = launch_state_pass(e, a, e->stream, 1, -1, sane)) return rc;
    }
    if (e->extras_on) {
        evaluate_extras_kernel<<<(unsigned)((states + 127) / 128), 128, 0, e->stream>>>(e->robot, e->sdf, e->extras, d_theta, num_trajectories, num_steps, d_cost);
        e->launch_count++;
        if (int rc = check_launch(e, "evaluate_extras_kernel")) return rc;
    }
    if (state_costs) CUDA_TRY(e, cudaMemcpyAsync(state_costs, d_cost, sizeof(double) * states, cudaMemcpyDeviceToHost, e->stream));
    if (verdicts) CUDA_TRY(e, cudaMemcpyAsync(verdicts, d_verdict, states, cudaMemcpyDeviceToHost, e->stream));
    if (validity) CUDA_TRY(e, cudaMemcpyAsync(validity, d_valid, num_trajectories, cudaMemcpyDeviceToHost, e->stream));
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    resolve_profile(e);
    return STOMP_B200_OK;
}

int stomp_b200_sphere_centres(stomp_b200_engine* e, const double* q, int32_t n, double* centres)
{
    if (!e || !q || !centres || n < 1) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_chain || !e->have_spheres) return fail(e, STOMP_B200_ERR_NOT_READY, "chain and spheres must be set first");
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    double* d_q = nullptr; double* d_c = nullptr;
    const size_t out_count = (size_t)n * e->robot.num_spheres * 3;
    CUDA_TRY(e, cudaMalloc(&d_q, sizeof(double) * n * e->D));
    cudaError_t err = cudaMalloc(&d_c, sizeof(double) * out_count);
    if (err == cudaSuccess) err = cudaMemcpyAsync(d_q, q, sizeof(double) * n * e->D, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) {
        sphere_centres_kernel<<<(n + 127) / 128, 128, 0, e->stream>>>(e->robot, d_q, n, d_c);
        e->launch_count++;
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaMemcpyAsync(centres, d_c, sizeof(double) * out_count, cudaMemcpyDeviceToHost, e->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    cudaFree(d_q); cudaFree(d_c);
    if (err != cudaSuccess) { e->last_error = std::string("sphere_centres: ") + cudaGetErrorString(err); return STOMP_B200_ERR_CUDA; }
    return STOMP_B200_OK;
}

int stomp_b200_comm_unique_id(void* id_out)
{
    if (!id_out) return STOMP_B200_ERR_INVALID_ARGUMENT;
    std::string err;
    if (!g_nccl.load(err)) return STOMP_B200_ERR_NCCL;
    static_assert(sizeof(ncclUniqueId) == STOMP_B200_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) return STOMP_B200_ERR_NCCL;
    std::memcpy(id_out, &id, sizeof(id));
    return STOMP_B200_OK;
}

int stomp_b200_comm_init(stomp_b200_engine* e, const void* id)
{
    if (!e || !id) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!g_nccl.load(e->last_error)) return STOMP_B200_ERR_NCCL;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, sizeof(uid));
    NCCL_TRY(e, g_nccl.CommInitRank(&e->comm, e->cfg.world_size, uid, e->cfg.rank));
    e->config_epoch++;
    if (e->cfg.shard_mode == 0 && e->cfg.world_size > 1) return setup_peer_exchange(e);
    return STOMP_B200_OK;
}

int32_t stomp_b200_exchange_kind(stomp_b200_engine* e, char* note, size_t note_capacity)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (note && note_capacity) std::snprintf(note, note_capacity, "%s", e->exchange_note.c_str());
    if (e->cfg.shard_mode != 0 || e->cfg.world_size <= 1 || !e->comm) return 0;
    return e->peer_ready ? 2 : 1;
}

int stomp_b200_set_profiling(stomp_b200_engine* e, int32_t on)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    join_side_stream(e);
    cudaStreamSynchronize(e->stream);
    resolve_profile(e);
    e->profiling = on != 0;
    return STOMP_B200_OK;
}

int stomp_b200_set_timeline(stomp_b200_engine* e, int32_t on)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    // begin stamps start at the largest value (atomicMin), end stamps at zero (atomicMax)
    std::vector<unsigned long long> init((size_t)kTimelineRing * kTimelineKernels * 2);
    for (size_t i = 0; i < init.size(); ++i) init[i] = (i & 1) ? 0ull : ~0ull;
    CUDA_TRY(e, cudaMemcpy(e->d_timeline, init.data(), sizeof(unsigned long long) * init.size(), cudaMemcpyHostToDevice));
    e->timeline_on = on != 0;
    e->timeline_count = 0;
    return STOMP_B200_OK;
}

int stomp_b200_get_timeline(stomp_b200_engine* e, int32_t max_iterations, double* begin_end_us, int32_t* num_iterations)
{
    if (!e || !begin_end_us || !num_iterations) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    const int n = (int)std::min<long long>(std::min<long long>(e->timeline_count, kTimelineRing), max_iterations);
    std::vector<unsigned long long> raw((size_t)kTimelineRing * kTimelineKernels * 2);
    CUDA_TRY(e, cudaMemcpy(raw.data(), e->d_timeline, sizeof(unsigned long long) * raw.size(), cudaMemcpyDeviceToHost));
    // oldest first; microseconds relative to the first stamp returned
    unsigned long long t0 = ~0ull;
    const long long first = e->timeline_count - n;
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < kTimelineKernels; ++k)
            t0 = std::min(t0, raw[((size_t)((first + i) % kTimelineRing) * kTimelineKernels + k) * 2]);
    for (int i = 0; i < n; ++i)
        for (int k = 0; k < kTimelineKernels; ++k) {
            const unsigned long long* r = raw.data() + ((size_t)((first + i) % kTimelineRing) * kTimelineKernels + k) * 2;
            const bool ran = r[0] != ~0ull && r[1] != 0ull;
            begin_end_us[((size_t)i * kTimelineKernels + k) * 2] = ran ? (double)(r[0] - t0) * 1e-3 : -1.0;
            begin_end_us[((size_t)i * kTimelineKernels + k) * 2 + 1] = ran ? (double)(r[1] - t0) * 1e-3 : -1.0;
        }
    *num_iterations = n;
    return STOMP_B200_OK;
}

int stomp_b200_kernel_stats(stomp_b200_engine* e, int32_t kernel, double* total_ms, int64_t* launches)
{
    if (!e || kernel < 0 || kernel >= STOMP_B200_KERNEL_COUNT) return STOMP_B200_ERR_INVALID_ARGUMENT;
    cudaStreamSynchronize(e->stream);
    resolve_profile(e);
    if (total_ms) *total_ms = e->kernel_ms[kernel];
    if (launches) *launches = e->kernel_launches[kernel];
    return STOMP_B200_OK;
}

int stomp_b200_reset_kernel_stats(stomp_b200_engine* e)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    cudaStreamSynchronize(e->stream);
    resolve_profile(e);
    for (int k = 0; k < STOMP_B200_KERNEL_COUNT; ++k) { e->kernel_ms[k] = 0; e->kernel_launches[k] = 0; }
    return STOMP_B200_OK;
}

int64_t stomp_b200_launch_count(const stomp_b200_engine* e) { return e ? e->launch_count : 0; }
int64_t stomp_b200_graph_replays(const stomp_b200_engine* e) { return e ? e->graph_launches : 0; }

int stomp_b200_timer_begin(stomp_b200_engine* e)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    if (e->peer_ready) {
        // the ranks of a sharded engine start the timed region together: a device-side barrier over the mailboxes, so that
        // no rank's bracket contains another rank's head start
        peer_barrier_kernel<<<1, 32, 0, e->stream>>>(e->px, ++e->barrier_ticket);
        e->launch_count++;
        if (int rc = check_launch(e, "peer_barrier_kernel")) return rc;
    }
    CUDA_TRY(e, cudaEventRecord(e->timer_a, e->stream));
    e->timer_armed = true;
    e->timer_end_recorded = false;
    return STOMP_B200_OK;
}

int stomp_b200_timer_end(stomp_b200_engine* e, double* elapsed_ms)
{
    if (!e || !elapsed_ms) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (int rc = join_side_stream(e)) return rc;
    // stomp_b200_run has put the end event behind its last kernel already (every call since timer_begin re-records it);
    // other call sequences (solve, iterate) end the region here
    if (!e->timer_end_recorded) CUDA_TRY(e, cudaEventRecord(e->timer_b, e->stream));
    e->timer_armed = false;
    e->timer_end_recorded = false;
    CUDA_TRY(e, cudaEventSynchronize(e->timer_b));
    float ms = 0.f;
    CUDA_TRY(e, cudaEventElapsedTime(&ms, e->timer_a, e->timer_b));
    *elapsed_ms = ms;
    return STOMP_B200_OK;
}

int stomp_b200_synchronize(stomp_b200_engine* e)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    CUDA_TRY(e, cudaSetDevice(e->cfg.device));
    if (int rc = join_side_stream(e)) return rc;
    CUDA_TRY(e, cudaStreamSynchronize(e->stream));
    resolve_profile(e);
    return STOMP_B200_OK;
}

}  // extern "C"

// ---- the run-time specialised state kernel (state_codegen.hpp) ------------------------------------------
int32_t stomp_b200_state_kernel_kind(stomp_b200_engine* e, char* note, size_t note_capacity)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_chain || !e->have_spheres || !e->have_sdf) return fail(e, STOMP_B200_ERR_NOT_READY, "chain, spheres and SDF come first");
    if (cudaSetDevice(e->cfg.device) != cudaSuccess) return fail(e, STOMP_B200_ERR_CUDA, "cudaSetDevice");
    resolve_state_kernel(e);
    if (note && note_capacity) {
        std::string text = e->spec ? ("specialised, " + std::to_string(e->spec->registers) + " registers") : ("generic: " + e->spec_note);
        if (e->self_pairs.n > 0) {
            resolve_self_kernel(e);
            text = "self-collision kernel (" + std::to_string(e->self_pairs.n) + " sphere pairs), " +
                   (e->spec_self ? "pair rule inside the specialised kernel (FP32 bands, FP64 where undecided), " + std::to_string(e->spec_self->registers) + " registers"
                                 : "generic FK: " + e->spec_self_note);
        }
        std::snprintf(note, note_capacity, "%s", text.c_str());
    }
    if (e->self_pairs.n > 0) return 2;
    return e->spec ? 1 : 0;
}

int stomp_b200_state_kernel_source(stomp_b200_engine* e, char* buffer, size_t capacity, size_t* needed)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (!e->have_chain || !e->have_spheres) return fail(e, STOMP_B200_ERR_NOT_READY, "chain and spheres come first");
    // the source of the kernel this engine launches; for an engine on the generic kernel, what would be generated
    const std::string src = (e->spec_resolved && e->spec) ? e->spec->source : codegen::generate_state_kernel_source(e->robot, state_kernel_options(e));
    if (needed) *needed = src.size() + 1;
    if (buffer && capacity) std::snprintf(buffer, capacity, "%s", src.c_str());
    return STOMP_B200_OK;
}

// Needs no device: generates the kernel for a synthetic structure that exercises every template branch (all axis
// kinds, fixed rotation, prismatic joint, chain restart, every zero mask, wide index) and compiles it to an
// sm_100a cubin with NVRTC.  The "does the generated code build" check of __graft_entry__.build().
int stomp_b200_codegen_selftest(char* log, size_t log_capacity)
{
    RobotParams r;
    std::memset(&r, 0, sizeof r);
    r.num_joints = 8;
    const int kinds[8] = {kAxisZ, kAxisY, kAxisX, kAxisNegX, kAxisNegY, kAxisNegZ, kAxisGeneral, kAxisZ};
    int sph = 0;
    for (int d = 0; d < 8; ++d) {
        JointParams& j = r.joint[d];
        j.axis_kind = kinds[d];
        j.o_mask = d & 7;
        j.fixed_rot_identity = (d == 3) ? 0 : 1;
        j.prismatic = (d == 7) ? 1 : 0;
        j.parent = (d == 0 || d == 4) ? -1 : d - 1;
        r.sphere_begin[d] = sph;
        for (int k = 0; k < (d % 3) + 1; ++k) r.sphere[sph++].mask = (d + k) & 7;
    }
    for (int d = 8; d <= STOMP_B200_MAX_DIMS; ++d) r.sphere_begin[d] = sph;
    r.num_spheres = sph;
    std::string all_log, err;
    int rc = STOMP_B200_OK;
    for (int wide = 0; wide < 2 && rc == STOMP_B200_OK; ++wide) {
        std::vector<char> cubin;
        std::string clog;
        codegen::StateKernelOptions opt;
        opt.wide_index = wide != 0;
        opt.magic_floor = wide == 0;
        opt.inside_grid = wide == 0;
        const std::string src = codegen::generate_state_kernel_source(r, opt);
        if (!codegen::compile_to_cubin(src, cubin, clog, err)) {
            all_log += err;
            rc = STOMP_B200_ERR_CUDA;
        } else {
            // both chains of the synthetic structure start with a sphere at the joint's origin: evaluated by stomp_b200_static_spheres
            const size_t at = src.find(" static spheres\n");
            const size_t from = at == std::string::npos ? at : src.rfind("// ", at);
            const std::string statics = from == std::string::npos ? std::string("no static spheres") : src.substr(from + 3, at - from - 3) + " static spheres";
            all_log += "ok: " + std::to_string(cubin.size()) + " byte cubin (" + codegen::cache().nvrtc.where + "), " + statics + " " + clog + "\n";
        }
    }
    if (rc == STOMP_B200_OK) {      // the same walk with the sphere-pair rule inside: every sphere of the first chain against every one of the second
        codegen::SelfPairStructure sp;
        std::vector<int> link_of((size_t)sph, 0);
        for (int d = 0; d < 8; ++d) for (int k = r.sphere_begin[d]; k < r.sphere_begin[d + 1]; ++k) link_of[k] = d;
        for (int i = 0; i < r.sphere_begin[4]; ++i)
            for (int j = r.sphere_begin[4]; j < sph; ++j) {
                const int la = link_of[i], lb = link_of[j];
                if (sp.blocks.empty() || sp.blocks.back().la != la || sp.blocks.back().lb != lb) sp.blocks.push_back({la, lb, (int)sp.i.size(), (int)sp.i.size()});
                sp.i.push_back(i); sp.j.push_back(j);
                sp.blocks.back().end = (int)sp.i.size();
            }
        sp.blocks.push_back({7, 7, (int)sp.i.size(), (int)sp.i.size() + 1});      // a pair inside one link: no cull
        sp.i.push_back(sph - 2); sp.j.push_back(sph - 1);
        std::vector<char> cubin;
        std::string clog;
        codegen::StateKernelOptions opt;
        opt.magic_floor = true; opt.inside_grid = true; opt.no_tail = true; opt.self = &sp;
        if (!codegen::compile_to_cubin(codegen::generate_state_kernel_source(r, opt), cubin, clog, err)) {
            all_log += err;
            rc = STOMP_B200_ERR_CUDA;
        } else {
            all_log += "ok (pair rule, " + std::to_string(sp.i.size()) + " pairs): " + std::to_string(cubin.size()) + " byte cubin " + clog + "\n";
        }
    }
    if (log && log_capacity) std::snprintf(log, log_capacity, "%s", all_log.c_str());
    return rc;
}

// Stomp::setCostCumulation (reference src/planners/stomp/src/Stomp.cpp:356-359): 1 = costs summed over the trajectory
// (the default, PolicyImprovement.cpp:56), 0 = costs and probabilities per time step.  Takes effect at the next iteration.
int stomp_b200_set_cost_cumulation(stomp_b200_engine* e, int32_t use_cumulative_costs)
{
    if (!e) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (use_cumulative_costs < 0 || use_cumulative_costs > 2) return STOMP_B200_ERR_INVALID_ARGUMENT;
    if (use_cumulative_costs != 1) {
        if (e->cfg.world_size > 1 || e->reuse_possible)
            return fail(e, STOMP_B200_ERR_UNSUPPORTED, "per-time-step costs are built for one GPU without rollout reuse");
        CUDA_TRY(e, cudaSetDevice(e->cfg.device));
        LoopParams& b = e->base;
        const size_t Q = e->Q, T = e->T, D = e->D, S = e->slots, GS = e->gslots;
        if (!b.control_costs) { if (int rc = dev_alloc(e, &b.control_costs, Q * S * D * T)) return rc; }
        if (!b.pt_prob) { if (int rc = dev_alloc(e, &b.pt_prob, Q * GS * D * T)) return rc; }
        if (!b.pt_minden) { if (int rc = dev_alloc(e, &b.pt_minden, Q * D * 2)) return rc; }
        if (use_cumulative_costs == 2 && !b.pt_cum) { if (int rc = dev_alloc(e, &b.pt_cum, Q * S * D * T)) return rc; }
    }
    e->cfg.use_cumulative_costs = use_cumulative_costs;
    e->config_epoch++;
    return STOMP_B200_OK;
}
