/*
 * stomp_b200.h — C ABI of the B200-native STOMP rollout loop.
 *
 * Drop-in boundary for the hot path of rock-planning/motion_planners: everything that
 * stomp::Stomp::runSingleIteration does per iteration (reference src/planners/stomp/src/Stomp.cpp:274-301)
 * — PolicyImprovement::generateRollouts, the Task::execute rollout cost, computeRolloutCumulativeCosts /
 * computeRolloutProbabilities and computeParameterUpdates / CovariantMovementPrimitive::updateParameters —
 * runs in hand-written sm_100a CUDA kernels behind these entry points.  The reference has no FFI of its
 * own (it is one C++ process); these are the calls our StompPlanner (include/wrapper/stomp/StompPlanner.hpp,
 * same public API as reference src/planners/include/wrapper/stomp/StompPlanner.hpp:15-89) makes where the
 * reference's StompPlanner::solve (src/planners/src/wrappers/stomp/StompPlanner.cpp:65-174) drives
 * stomp::Stomp.  INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns an int status (0 = ok, negative =
 * error, never throws or aborts); all host buffers are caller-owned, row-major, FP64 unless stated;
 * one engine <-> one host thread <-> one GPU.  There is NO CPU fallback: without a CUDA device
 * stomp_b200_create fails with STOMP_B200_ERR_NO_DEVICE.
 *
 * Index names: Q queries held by this engine, K' = rollouts used in the current update (generated +
 * reused + the appended noise-less one), G = rollouts generated in the current iteration, D joints,
 * T time steps, N = T + 12 (TRAJECTORY_PADDING = 6 on both sides, reference StompUtils.hpp:57), S spheres.
 */
#ifndef STOMP_B200_H_
#define STOMP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STOMP_B200_ABI_VERSION 1
#define STOMP_B200_MAX_DIMS 32      /* joints per planning group */
#define STOMP_B200_MAX_SPHERES 128  /* collision spheres */
#define STOMP_B200_MAX_TIME_STEPS 256

enum stomp_b200_status {
    STOMP_B200_OK = 0,
    STOMP_B200_ERR_INVALID_ARGUMENT = -1,
    STOMP_B200_ERR_NO_DEVICE = -2,       /* no CUDA device / driver: the product path has no CPU fallback */
    STOMP_B200_ERR_CUDA = -3,            /* a CUDA call failed; see stomp_b200_last_error */
    STOMP_B200_ERR_NOT_READY = -4,       /* chain / spheres / SDF / policy / begin_solve missing */
    STOMP_B200_ERR_UNSUPPORTED = -5,     /* valid in the reference, not built yet (listed in DESIGN.md) */
    STOMP_B200_ERR_NCCL = -6,
    STOMP_B200_ERR_OUT_OF_MEMORY = -7
};

typedef struct stomp_b200_engine stomp_b200_engine;

/* Mirrors stomp::StompConfig (reference src/planners/stomp/include/stomp/StompConfig.hpp:19-42) plus the
 * switches the reference hard-codes in PolicyImprovement's constructor (PolicyImprovement.cpp:52-58). */
typedef struct stomp_b200_config {
    int32_t abi_version;                 /* STOMP_B200_ABI_VERSION */
    int32_t num_time_steps;              /* T  (num_time_steps_) */
    int32_t num_dimensions;              /* D  (num_dimensions_) */
    int32_t min_rollouts;                /* min_rollouts_ */
    int32_t max_rollouts;                /* max_rollouts_ */
    int32_t num_rollouts_per_iteration;  /* num_rollouts_per_iteration_ */
    int32_t num_queries;                 /* Q_total: independent planning queries (batch mode); 1 = the reference */
    double movement_duration;            /* movement_duration_ */
    double control_cost_weight;          /* control_cost_weight_ */
    double min_cost_improvement;         /* min_cost_improvement_ (stop rule, StompPlanner.cpp:117) */
    double noise_stddev[STOMP_B200_MAX_DIMS];
    double noise_decay[STOMP_B200_MAX_DIMS];
    double noise_min_stddev[STOMP_B200_MAX_DIMS];
    double derivative_weights[4];        /* position, velocity, acceleration, jerk; the reference task sets
                                            {0,0,1,0} for every joint and time step (OptimizationTask.cpp:32-33) */
    double cost_scaling_h;               /* 10.0 (PolicyImprovement.cpp:55) */
    int32_t use_noise_adaptation;        /* use_noise_adaptation_ */
    int32_t use_cumulative_costs;        /* 1 (PolicyImprovement.cpp:56): costs summed over the trajectory; 0 = per-time-step costs;
                                            2 = forward cumulation, cumulative_costs_(t) = sum_{t' >= t} (the variant commented out at
                                            :473-477).  0 and 2: one GPU, no rollout reuse */
    int32_t use_projection;              /* 0 (PolicyImprovement.cpp:57); 1 = M-matrix projected noise / update
                                            (PolicyImprovement.cpp:421-440,706,750-801); needs Rinv */
    int32_t per_timestep_minmax;         /* 0 = shipped global min/max; 1 = variant commented out at :518-528 (differs
                                            from 0 only with use_cumulative_costs == 0) */
    int32_t device;                      /* CUDA device ordinal */
    int32_t world_size;                  /* ranks (one per GPU) sharing this solve; 1 = single GPU */
    int32_t rank;
    int32_t shard_mode;                  /* 0: rollouts of one query sharded over ranks (needs stomp_b200_comm_init);
                                            1: queries sharded over ranks, no collective */
    int32_t keep_debug_tensors;          /* 1: keep per-(k,d,t) control costs, unit noise and epsilon for read-back */
    uint64_t seed;                       /* Philox seed of the on-device sampler */
} stomp_b200_config;

void stomp_b200_default_config(stomp_b200_config* cfg);
int stomp_b200_abi_version(void);
const char* stomp_b200_status_string(int status);
/* text of the last failure on this engine (CUDA / NCCL error strings included); never NULL */
const char* stomp_b200_last_error(const stomp_b200_engine* e);

/* ---- lifecycle --------------------------------------------------------------------------------------
 * create: what StompPlanner::initializePlanner + `new OptimizationTask` set up
 * (StompPlanner.cpp:15-38, OptimizationTask.cpp:8-44), on the device. */
int stomp_b200_create(const stomp_b200_config* cfg, stomp_b200_engine** out);
int stomp_b200_destroy(stomp_b200_engine* e);

/* ---- robot + scene: replaces robot_model::RobotModel::updateJointGroup + isStateValid ------------------
 * (call sites OptimizationTask.cpp:190,192).  Joints are URDF joints in chain order
 * (reference test/data/kuka_iiwa.urdf:162-210): origin xyz / rpy, axis, limits.  parent[d] is d-1, or -1
 * for a joint that hangs off the fixed base frame (a second arm restarts the chain that way).
 * prismatic may be NULL (all revolute).  lower/upper are what OptimizationTask::filter clamps to
 * (OptimizationTask.cpp:85-106). */
int stomp_b200_set_chain(stomp_b200_engine* e, int32_t num_joints, const double* origin_xyz /*[D][3]*/,
                         const double* origin_rpy /*[D][3]*/, const double* axis /*[D][3]*/,
                         const int32_t* parent /*[D]*/, const int32_t* prismatic /*[D] or NULL*/,
                         const double* lower /*[D]*/, const double* upper /*[D]*/);
/* link[s] = joint whose child link carries sphere s; must be sorted ascending (grasped-object spheres are
 * spheres on the tip link). */
int stomp_b200_set_spheres(stomp_b200_engine* e, int32_t num_spheres, const int32_t* link /*[S]*/,
                           const double* centre_xyz /*[S][3]*/, const double* radius /*[S]*/);
/* FP32 signed distance grid, x fastest: grid[(z*ny + y)*nx + x]; origin = min corner of voxel (0,0,0).
 * Nearest-voxel lookup, coordinates clamped to the grid.  The grid is copied to the device. */
int stomp_b200_set_sdf(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                       const float* grid);

/* ---- environment -> distance field, built on the device (SURVEY.md 8f rank 2) --------------------------------
 * The reference hands its world to FCL as collision objects: primitives, meshes, an octomap
 * (src/MotionPlanners.cpp:162-173 assignOctomapPlanningScene / updateOctomap, :416-495 handleCollisionObjectInWorld /
 * handleGraspObject; include/motion_planners/Config.hpp:14-35).  Here they become the distance field the state kernel
 * gathers from, without a host grid or a host-to-device copy of it:
 *   primitives: kind[i] 0 = sphere (size[i][0] = radius), 1 = box (size[i] = half extents), 2 = cylinder along z
 *     (size[i] = radius, half height) — the reference's PrimitiveObject types box / cylinder / sphere; exact signed distance of
 *     the union at every voxel centre origin + (i + 0.5) * voxel_size, FP64, rounded to binary32;
 *   occupancy [nz][ny][nx] uint8 (a voxelised mesh, or the leaves of an octomap at the grid's resolution): exact
 *     Euclidean distance transform, centre to centre, positive outside the occupied set and negative inside.
 * get_sdf copies the grid back (tests / inspection); any output may be NULL. */
int stomp_b200_build_sdf_primitives(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                                    int32_t num_primitives, const int32_t* kind /*[n]*/, const double* centre /*[n][3]*/,
                                    const double* size /*[n][3]*/);
int stomp_b200_build_sdf_occupancy(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                                   const uint8_t* occupied /*[nz][ny][nx]*/);
/* The general scene: the union of
 *   a triangle mesh (the reference's MESH model objects; triangles [n][3 vertices][xyz] in the grid's frame), voxelised
 *     conservatively on the device (a voxel is occupied when its cube touches a triangle); solid != 0 also fills the
 *     interior of closed meshes (free voxels the grid's boundary cannot reach);
 *   octomap leaves (occupied cubes: centre [m][3] and edge length [m]; a voxel is occupied when its centre lies in a leaf);
 *   an occupancy grid (may be NULL);
 * followed by the exact distance transform of stomp_b200_build_sdf_occupancy.  Any of the three parts may be empty. */
int stomp_b200_build_sdf_scene(stomp_b200_engine* e, const int32_t dims[3], const double origin[3], double voxel_size,
                               int32_t num_triangles, const double* triangles /*[n][3][3] or NULL*/, int32_t solid,
                               int32_t num_leaves, const double* leaf_centres /*[m][3] or NULL*/,
                               const double* leaf_sizes /*[m] or NULL*/, const uint8_t* occupied /*[nz][ny][nx] or NULL*/);
int stomp_b200_get_sdf(stomp_b200_engine* e, float* out, size_t count, int32_t dims_out[3], double origin_out[3],
                       double* voxel_size_out);

/* ---- scenes: one distance field each; every local query reads the field of its scene ----------------------------------
 * A batch can hold queries in different worlds (datasets over many environments, benchmark suites of many scenes, a fleet
 * of cells with their own obstacles).  An engine starts with scene 0, which every query uses; an engine that never calls
 * the two functions below behaves exactly as before.
 * select_scene: set_sdf, build_sdf_primitives / _occupancy / _scene, get_sdf and evaluate_states act on `scene` from now
 * on.  Indices are dense: 0 <= scene <= current number of scenes (selecting that number creates an empty scene).
 *   - A scene has its own dims, origin and voxel size.
 *   - Rebuilding a scene, or reassigning queries to scenes, between solves takes effect from the next iteration, in loops
 *     replayed from CUDA graphs too.
 *   - begin_solve, iterate, run and solve return STOMP_B200_ERR_NOT_READY while a local query's scene has no field
 *     (stomp_b200_last_error names the query and the scene).
 *   - A bad query range, a negative scene or a scene that does not exist: STOMP_B200_ERR_INVALID_ARGUMENT.
 *   - Query indices are local, as for policies: under query sharding each rank holds the scenes its caller gives it.
 * The Philox noise of a query does not depend on its scene: a batch spread over several scenes draws what the same batch
 * in one scene draws. */
int stomp_b200_select_scene(stomp_b200_engine* e, int32_t scene);
/* scene[i] for local queries first_query .. first_query + count - 1 (query-major like stomp_b200_set_policies). */
int stomp_b200_set_query_scenes(stomp_b200_engine* e, int32_t first_query, int32_t count, const int32_t* scene);

/* ---- policy: the host-computed products of CovariantMovementPrimitive::initialize ----------------------
 * (CovariantMovementPrimitive.cpp:57-74,136-301; computed by stomp_b200_host_policy below or by the
 * C++ stomp::CovariantMovementPrimitive in include/stomp/).  R = control_costs_, Rinv = inv_control_costs_,
 * L = chol(Rinv) (MultivariateGaussian.hpp:81); identical for every joint and query.  Rinv may be NULL
 * unless use_projection (then the projection matrix and its inverse are formed from it here,
 * PolicyImprovement::preComputeProjectionMatrices). */
int stomp_b200_set_control_cost_matrices(stomp_b200_engine* e, const double* R /*[T][T]*/,
                                         const double* Rinv /*[T][T] or NULL*/, const double* L /*[T][T]*/);
/* per query (local index): parameters_all_ [D][N] (padding = start / goal) and
 * min_control_cost_parameters_free_ [D][T] */
int stomp_b200_set_policy(stomp_b200_engine* e, int32_t query, const double* parameters_all /*[D][N]*/,
                          const double* min_control_cost /*[D][T]*/);
/* the same for `count` consecutive local queries starting at first_query, arrays query-major: one pair of copies for a
 * whole batch of planning requests (StompPlanner::setStartGoalTrajectory of every request of a batch) */
int stomp_b200_set_policies(stomp_b200_engine* e, int32_t first_query, int32_t count,
                            const double* parameters_all /*[count][D][N]*/, const double* min_control_cost /*[count][D][T]*/);

/* Host-side (CPU, one-time per query shape) CovariantMovementPrimitive::initialize +
 * computeLinearControlCosts + (optionally) setToMinControlCost.  initial_all [D][N] is the padded
 * initial trajectory (OptimizationTask::updateTrajectory, OptimizationTask.cpp:46-66).  Any output may
 * be NULL.  No device needed. */
int stomp_b200_host_policy(int32_t num_time_steps, int32_t num_dimensions, double movement_duration,
                           const double derivative_weights[4], const double* initial_all /*[D][N]*/,
                           int32_t set_to_min_control_cost, double* R, double* Rinv, double* L,
                           double* parameters_all_out /*[D][N]*/, double* min_control_cost_out /*[D][T]*/);
/* OptimizationTask::updateTrajectory (OptimizationTask.cpp:46-66): linear interpolation + padding */
int stomp_b200_host_initial_trajectory(int32_t num_time_steps, int32_t num_dimensions, const double* start,
                                       const double* goal, double* initial_all /*[D][N]*/);

/* ---- the loop: StompPlanner::solve (StompPlanner.cpp:65-174) --------------------------------------------
 * begin_solve = `new stomp::Stomp` + Stomp::initialize (Stomp.cpp:56-94): resets the rollout bookkeeping,
 * the adapted noise and the noise-less rollout. */
int stomp_b200_begin_solve(stomp_b200_engine* e);

/* One Stomp::runSingleIteration (Stomp.cpp:274-301) for every query of the engine, then the wrapper's
 * bookkeeping (StompPlanner.cpp:107-118).  Synchronous.  Noise sources, first non-NULL wins:
 *   unit_noise [Q][G][D][T]: the output of MultivariateGaussian::sample (L*eps, zero mean) — parity mode;
 *   epsilon    [Q][G][D][T]: standard normals, pushed through L on the device;
 *   neither: Philox4x32-10 normals generated on the device.
 * G = stomp_b200_next_num_generated(e).  Outputs (any may be NULL), per query:
 * noiseless_total_cost (getNoiselessRolloutTotalCost), noiseless_valid (last_noiseless_rollout_valid_),
 * stop (1 when the stop rule of StompPlanner.cpp:117 fired in this or an earlier iteration). */
int stomp_b200_iterate(stomp_b200_engine* e, int32_t iteration, const double* unit_noise, const double* epsilon,
                       double* noiseless_total_cost /*[Q]*/, uint8_t* noiseless_valid /*[Q]*/, int32_t* stop /*[Q]*/);
int32_t stomp_b200_next_num_generated(const stomp_b200_engine* e);

/* num_iterations passes of the loop body with the on-device sampler, queued without host round trips;
 * a query whose stop rule fired is frozen (honour_stop != 0) exactly as `break` leaves it in the
 * reference.  Returns after the last kernel finished. */
int stomp_b200_run(stomp_b200_engine* e, int32_t first_iteration, int32_t num_iterations, int32_t honour_stop);

/* The whole iteration loop of StompPlanner::solve (StompPlanner.cpp:96-141) on the device: up to max_iterations
 * iterations with the on-device sampler and the stop rule honoured per query (a stopped query is frozen exactly where
 * the reference's `break` leaves it: parameters, noise-less cost, iteration count).  The host queues iterations one
 * ahead of two progress words per query (noise-less rollouts recorded, stopped) that the device writes into mapped pinned
 * host memory, stops queueing once every query has stopped and synchronises once, at the end; that read-back brings the
 * per-query scalars and the solution rows into pinned mirrors, so that a stomp_b200_finish_solve straight after makes no
 * device call.  Rollout-sharded engines (every rank has to queue the same iterations) look at the stop flags every
 * poll_every iterations instead (<= 0: 8; one pinned read-back and one synchronisation per poll).  Iterations queued past
 * a query's stop are no-ops for it.  iterations_run (may be NULL) = iterations queued; the per-query counts come from
 * stomp_b200_finish_solve. */
int stomp_b200_solve(stomp_b200_engine* e, int32_t max_iterations, int32_t poll_every, int32_t* iterations_run);

/* Stomp::setCostCumulation (stomp/src/Stomp.cpp:356-359): 1 = costs summed over the trajectory (the default), 0 = costs
 * and probabilities per time step (PolicyImprovement.cpp:473-481), 2 = forward cumulation (cost-to-go, :473-477).  0 and 2
 * are built for one GPU without rollout reuse, else
 * STOMP_B200_ERR_UNSUPPORTED.  Also settable at creation (stomp_b200_config::use_cumulative_costs). */
int stomp_b200_set_cost_cumulation(stomp_b200_engine* e, int32_t use_cumulative_costs);

/* end of StompPlanner::solve (:148-173): solution = parameters_all_[d][6+t] (the LAST parameters, not the
 * best noise-less ones); status 1 = PATH_FOUND, 0 = NO_PATH_FOUND; iterations_used = getNumOfIterationsUsed. */
int stomp_b200_finish_solve(stomp_b200_engine* e, double* solution /*[Q][D][T]*/, int32_t* status /*[Q]*/,
                            int32_t* iterations_used /*[Q]*/, double* noiseless_total_cost /*[Q]*/);

/* ---- read-backs of the state of the last iteration (parity tests; stomp::Rollout fields,
 * PolicyImprovement.hpp:49-68).  Leading dimension is always the local query. */
enum stomp_b200_tensor {
    STOMP_B200_ROLLOUTS = 0,            /* parameters_noise_          [Q][K'][D][T] */
    STOMP_B200_NOISE = 1,               /* noise_                     [Q][K'][D][T] */
    STOMP_B200_STATE_COSTS = 2,         /* state_costs_               [Q][K'][T]    */
    STOMP_B200_VERDICTS = 3,            /* 1 = in collision, uint8    [Q][K'][T]    */
    STOMP_B200_CONTROL_COSTS = 4,       /* control_costs_             [Q][K'][D][T] (keep_debug_tensors) */
    STOMP_B200_CUMULATIVE_COSTS = 5,    /* cumulative_costs_[d](0)    [Q][K'][D]  (cumulative mode: constant over t) */
    STOMP_B200_FULL_COSTS = 6,          /* full_costs_                [Q][K'][D]    */
    STOMP_B200_TOTAL_COST = 7,          /* total_cost_                [Q][K']       */
    STOMP_B200_PROBABILITIES = 8,       /* probabilities_             [Q][K'][D][T] */
    STOMP_B200_FULL_PROBABILITIES = 9,  /* full_probabilities_        [Q][K'][D]    */
    STOMP_B200_UPDATES = 10,            /* parameter_updates_[d].row(0) [Q][D][T]   */
    STOMP_B200_PARAMETERS = 11,         /* policy parameters (free)   [Q][D][T]     */
    STOMP_B200_PARAMETERS_ALL = 12,     /* parameters_all_            [Q][D][N]     */
    STOMP_B200_STDDEVS = 13,            /* adapted_stddevs_           [Q][D]        */
    STOMP_B200_NOISELESS_STATE_COSTS = 14, /* noiseless_rollout_.state_costs_ [Q][T] */
    STOMP_B200_NOISELESS_CONTROL_COSTS = 15, /*                       [Q][D][T]     */
    STOMP_B200_UNIT_NOISE = 16,         /* L*eps of the generated rollouts [Q][G][D][T] (keep_debug_tensors) */
    STOMP_B200_EPSILON = 17,            /* eps of the generated rollouts   [Q][G][D][T] (keep_debug_tensors) */
    STOMP_B200_ROLLOUT_VALIDITY = 18,   /* execute()'s validity, uint8     [Q][G]       */
    STOMP_B200_NOISE_PROJECTED = 19,    /* noise_projected_ = M * noise_   [Q][K'][D][T] (use_projection) */
    STOMP_B200_ROLLOUTS_PROJECTED = 20  /* parameters_noise_projected_     [Q][K'][D][T] (configurations with rollout reuse) */
};
int stomp_b200_num_rollouts(const stomp_b200_engine* e, int32_t* num_rollouts /*K'*/, int32_t* num_generated /*G*/);
/* copies the tensor to host memory; out_bytes must equal its size */
int stomp_b200_get_tensor(stomp_b200_engine* e, int32_t tensor, void* out, size_t out_bytes);

/* ---- the cost kernel on its own (Task::execute for arbitrary trajectories; also what
 * MotionPlanners::checkStartState / checkGoalState need with K = 1, T = 1) -------------------------------
 * theta [K][D][Tq] host; outputs host, any may be NULL. */
int stomp_b200_evaluate_states(stomp_b200_engine* e, const double* theta, int32_t num_trajectories,
                               int32_t num_steps, double* state_costs /*[K][Tq]*/, uint8_t* verdicts /*[K][Tq]*/,
                               uint8_t* validity /*[K]*/);
/* ---- self collision (the "self" half of robot_model's isStateValid; which link pairs are checked is the host's
 * business: the reference's SRDF lists the disabled ones, test/data/kuka_iiwa.srdf:46-70).  pairs [num_pairs][2] are
 * indices into the sphere list of stomp_b200_set_spheres; a state is then in collision when a sphere is inside an
 * obstacle OR |c_i - c_j|^2 < (r_i + r_j)^2 for a listed pair.  Applies to the loop, the noise-less rollout and
 * stomp_b200_evaluate_states.  num_pairs == 0 switches the check off (the default); stomp_b200_set_spheres clears the
 * list.  While a list is set the state kernel is the generic-FK self-collision kernel
 * (stomp_b200_state_kernel_kind returns 2). */
int stomp_b200_set_self_collision(stomp_b200_engine* e, int32_t num_pairs, const int32_t* pairs /*[num_pairs][2]*/);

/* ---- alternative state costs (SURVEY.md 8f rank 4; both off by default = the reference's shipped 0 / 1 collision cost).
 * smooth obstacle cost: the state cost becomes smooth_weight * sum_s max(0, (r_s + smooth_margin) - d_s) over the link
 *   spheres — it grows with the penetration into the clearance band instead of jumping to 1 (the non-boolean obstacles of
 *   the reference's stomp/test/stomp_2d_test.cpp:337-363, carried over to spheres and a distance field);
 * joint-constraint cost: OptimizationTask::computeJointsConstraintCost / getConstrainDifference
 *   (src/planners/src/wrappers/stomp/OptimizationTask.cpp:206-237; its call at :169-172 is commented out in the reference):
 *   + weight * sum_d max(0, |value_d - q_d| - tolerance_d) on every time step.
 * The verdicts / validity stay the binary collision test.  Applies to the loop, the noise-less rollout and
 * stomp_b200_evaluate_states.  value / tolerance [D] may be NULL when use_joint_constraint == 0.  Works with rollout and query sharding (set it on every rank). */
int stomp_b200_set_cost_extras(stomp_b200_engine* e, int32_t use_smooth_cost, double smooth_margin, double smooth_weight,
                               int32_t use_joint_constraint, const double* value /*[D]*/, const double* tolerance /*[D]*/,
                               double joint_constraint_weight);

/* sphere centres in the world frame for n joint configurations q [n][D] -> [n][S][3] */
int stomp_b200_sphere_centres(stomp_b200_engine* e, const double* q, int32_t n, double* centres);

/* ---- the state kernel (FK + sphere / SDF verdicts) is specialised at run time to the robot's STRUCTURE (axis
 * kinds, zero masks, spheres per link) with NVRTC; numbers stay kernel parameters.  kind: 1 = specialised,
 * 0 = the generic CUDA kernel (libnvrtc missing, or STOMP_B200_STATES=generic); note says which / why.
 * source: the generated CUDA source for the engine's robot (needed includes the terminating NUL).
 * codegen_selftest needs no device: it generates and NVRTC-compiles a structure that uses every branch. */
int32_t stomp_b200_state_kernel_kind(stomp_b200_engine* e, char* note, size_t note_capacity);
int stomp_b200_state_kernel_source(stomp_b200_engine* e, char* buffer, size_t capacity, size_t* needed);
int stomp_b200_codegen_selftest(char* log, size_t log_capacity);

/* ---- multi-GPU (shard_mode 0): one engine per rank; rank 0 makes the id, the host side broadcasts it ---- */
#define STOMP_B200_COMM_ID_BYTES 128
int stomp_b200_comm_unique_id(void* id_out /*[128]*/);
int stomp_b200_comm_init(stomp_b200_engine* e, const void* id /*[128]*/);
/* How the two per-iteration exchanges of a rollout-sharded engine travel: 2 = peer-mapped mailboxes over NVLink, written
 * and awaited from inside the weights / update kernel (the default when cudaIpc works between the ranks); 1 = NCCL
 * all-gather + all-reduce (STOMP_B200_EXCHANGE=nccl, or the mailboxes could not be mapped: note says why); 0 = nothing is
 * exchanged (one GPU, or query sharding).  In mode 2 the rollout-indexed read-backs (costs, probabilities) of
 * stomp_b200_get_tensor are collective calls: every rank must ask for them in the same order. */
int32_t stomp_b200_exchange_kind(stomp_b200_engine* e, char* note, size_t note_capacity);

/* ---- measurement ----------------------------------------------------------------------------------- */
enum stomp_b200_kernel {
    STOMP_B200_KERNEL_SAMPLE = 0,       /* generateRollouts: L*eps contraction + mean shift + clamp */
    STOMP_B200_KERNEL_COST = 1,         /* rollout state cost: FK + sphere/SDF verdicts (the roofline kernel, 8D+4S+9 B/state) */
    STOMP_B200_KERNEL_WEIGHTS = 2,      /* computeRolloutProbabilities */
    STOMP_B200_KERNEL_UPDATE = 3,       /* probability-weighted sums + n^T R n */
    STOMP_B200_KERNEL_APPLY = 4,        /* updateParameters + noise adaptation + noise-less rollout */
    STOMP_B200_KERNEL_REUSE = 5,        /* importance sort + gather of reused rollouts */
    STOMP_B200_KERNEL_ROWS = 6,         /* control-cost stencil + n^T R n per (rollout, joint) row */
    STOMP_B200_KERNEL_COUNT = 7
};
/* when on, every launch of the kernels above is bracketed by CUDA events on the engine's stream */
int stomp_b200_set_profiling(stomp_b200_engine* e, int32_t on);
int stomp_b200_kernel_stats(stomp_b200_engine* e, int32_t kernel, double* total_ms, int64_t* launches);
int stomp_b200_reset_kernel_stats(stomp_b200_engine* e);
/* In-pipeline timeline: while on, every kernel stamps %globaltimer at its first CTA start and last CTA end;
 * get_timeline returns, oldest first, [iteration][8 kernels][begin, end] in microseconds relative to the first
 * stamp (-1 where a kernel did not run) for the last <= 64 iterations; kernels: 0 sample, 1 cost, 2 weights,
 * 3 update, 4 apply, 5 noise-less rollout, 6 reuse, 7 unused.  set_timeline(on) clears the ring. */
#define STOMP_B200_TIMELINE_KERNELS 8
int stomp_b200_set_timeline(stomp_b200_engine* e, int32_t on);
int stomp_b200_get_timeline(stomp_b200_engine* e, int32_t max_iterations, double* begin_end_us, int32_t* num_iterations);
/* total kernel launches issued by this engine since creation */
int64_t stomp_b200_launch_count(const stomp_b200_engine* e);
/* iterations that ran as one cudaGraphLaunch: steady-state iterations of the on-device-sampler loop (no rollout reuse, no
 * read-back tensors kept) of rollout shards and small problems are captured once and replayed; their kernels are counted in
 * stomp_b200_launch_count as usual.  Loops whose sampler fills the GPU are launched plainly instead: their sampler draws its
 * noise beside the previous iteration's update kernel (programmatic dependent launch), which a graph boundary would undo.
 * STOMP_B200_GRAPH=0 in the environment at stomp_b200_create switches the replay off, =2 replays those loops too. */
int64_t stomp_b200_graph_replays(const stomp_b200_engine* e);
/* device-side timing of a region on the engine's stream: begin waits for the stream, records an event and arms the timer;
 * the first stomp_b200_run inside the region moves that event to its own entry (the stream is idle in between), every
 * stomp_b200_run records the end event behind the last kernel it queues (before its own closing wait); without a run call
 * (solve, iterate) the region is begin .. end as called.  end waits for the end event and returns the milliseconds. */
int stomp_b200_timer_begin(stomp_b200_engine* e);
int stomp_b200_timer_end(stomp_b200_engine* e, double* elapsed_ms);
int stomp_b200_synchronize(stomp_b200_engine* e);

#ifdef __cplusplus
}
#endif
#endif /* STOMP_B200_H_ */
