/*
 * teb_b200.h — C-ABI of the B200-native Timed-Elastic-Band optimizer.
 *
 * This is the drop-in boundary for the hot path of rst-tu-dortmund/teb_local_planner:
 *   TebOptimalPlanner::optimizeTEB            src/optimal_planner.cpp:182-231
 *   TebOptimalPlanner::buildGraph/optimizeGraph/computeCurrentCost
 *                                             src/optimal_planner.cpp:323-366, 368-402, 1041-1094
 *   g2o SparseOptimizer + LM + CSparse        call sites src/optimal_planner.cpp:161-179, 385-387
 *   HomotopyClassPlanner::optimizeAllTEBs     src/homotopy_class_planner.cpp:466-493
 *   HomotopyClassPlanner::selectBestTeb       src/homotopy_class_planner.cpp:564-667
 *   TimedElasticBand::autoResize              src/timed_elastic_band.cpp:227-286
 *   HomotopyClassPlanner::calculateEquivalenceClass (HSignature / HSignature3d)
 *                                             include/teb_local_planner/homotopy_class_planner.hpp:46-63, h_signature.h
 *
 * Plain C, plain pointers and sizes, no torch / CUDA types in any signature.
 * All state is fp64 (the reference is fp64 throughout).
 *
 * Band storage ("pose records"): one band = n_cap records of 4 doubles
 *   rec[i] = { x_i, y_i, theta_i, dt_i }      dt_i = TimeDiff(i) connects pose i -> i+1
 * the last valid record (i = n-1) carries dt = 0.  Pose 0 and pose n-1 are fixed
 * during optimisation (timed_elastic_band.cpp:330,377), every dt is free.
 */
#ifndef TEB_B200_H
#define TEB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TEBGPU_OK                  0
#define TEBGPU_ERR_INVALID_ARG    -1
#define TEBGPU_ERR_CUDA           -2
#define TEBGPU_ERR_UNSUPPORTED    -3   /* an option outside what the kernels cover (e.g. unknown footprint model): fail loudly */
#define TEBGPU_ERR_CAPACITY       -4
#define TEBGPU_ERR_NO_DEVICE      -5

/* per-band status bits written to status[] */
#define TEB_STATUS_OPTIMIZED       1   /* optimizeTEB returned true (optimal_planner.cpp:220)      */
#define TEB_STATUS_TOO_FEW_POSES   2   /* sizePoses < min_samples guard (optimal_planner.cpp:377)   */
#define TEB_STATUS_CHOL_FAILED     4   /* at least one trial factorisation hit a pivot that is not a positive normal
                                          number (<= 0, subnormal, inf or NaN); a non-finite solution is not a failure */
#define TEB_STATUS_NONFINITE       8   /* non-finite chi2 / lambda encountered                      */
#define TEB_STATUS_TERMINATED     16   /* LM returned Terminate in the last optimizeGraph call      */
#define TEB_STATUS_DISABLED       32   /* optimization_activate == false / max_vel_x < 0.01          */
#define TEB_STATUS_CAPACITY       64   /* autoResize needed more than n_cap poses: band left unoptimised */
#define TEB_STATUS_BAD_INPUT     128   /* the band's scene holds an obstacle row the batch cannot describe (vertex range
                                          outside obst_vertices, unknown type): band left unoptimised */

/* robot_footprint_model.h: PointRobotFootprint :131, CircularRobotFootprint :205, TwoCirclesRobotFootprint :303,
 * LineRobotFootprint :439, PolygonRobotFootprint :635 */
enum { TEB_FOOTPRINT_POINT = 0, TEB_FOOTPRINT_CIRCULAR = 1, TEB_FOOTPRINT_TWO_CIRCLES = 2, TEB_FOOTPRINT_LINE = 3,
       TEB_FOOTPRINT_POLYGON = 4 };
/* obstacles.h: PointObstacle :305, CircularObstacle :447, LineObstacle :597, PillObstacle :746, PolygonObstacle :893 */
enum { TEB_OBST_POINT = 0, TEB_OBST_CIRCULAR = 1, TEB_OBST_LINE = 2, TEB_OBST_PILL = 3, TEB_OBST_POLYGON = 4 };
#define TEB_MAX_FOOTPRINT_VERTICES 16
enum { TEB_ROTDIR_NONE = 0, TEB_ROTDIR_LEFT = 1, TEB_ROTDIR_RIGHT = 2 };

/* POD mirror of the TebConfig fields read on the hot path
 * (include/teb_local_planner/teb_config.h:72-229, defaults :245-390). */
typedef struct TebParams {
  /* trajectory */
  double  dt_ref;
  double  dt_hysteresis;
  double  force_reinit_new_goal_dist;
  double  force_reinit_new_goal_angular;
  int32_t teb_autosize;
  int32_t min_samples;
  int32_t max_samples;
  int32_t exact_arc_length;
  int32_t via_points_ordered;
  int32_t allow_init_with_backwards_motion;
  int32_t global_plan_overwrite_orientation;
  int32_t _pad0;
  /* robot */
  double  max_vel_x;
  double  max_vel_x_backwards;
  double  max_vel_y;
  double  max_vel_trans;
  double  max_vel_theta;
  double  acc_lim_x;
  double  acc_lim_y;
  double  acc_lim_theta;
  double  min_turning_radius;
  /* footprint model (robot_footprint_model.h) */
  double  footprint_radius;        /* circular  */
  double  footprint_front_offset;  /* two circles */
  double  footprint_front_radius;
  double  footprint_rear_offset;
  double  footprint_rear_radius;
  int32_t footprint_type;
  int32_t footprint_vertex_count;  /* polygon: 1 .. TEB_MAX_FOOTPRINT_VERTICES (robot frame, not closed) */
  double  footprint_line[4];       /* line: start x, y, end x, y in the robot frame (robot_footprint_model.h:439) */
  double  footprint_vertices[2 * TEB_MAX_FOOTPRINT_VERTICES]; /* polygon: x0, y0, x1, y1, ... (:635) */
  /* obstacles */
  double  min_obstacle_dist;
  double  inflation_dist;
  double  dynamic_obstacle_inflation_dist;
  double  obstacle_association_force_inclusion_factor;
  double  obstacle_association_cutoff_factor;
  double  obstacle_proximity_ratio_max_vel;
  double  obstacle_proximity_lower_bound;
  double  obstacle_proximity_upper_bound;
  int32_t include_dynamic_obstacles;
  int32_t legacy_obstacle_association;
  int32_t obstacle_poses_affected;
  int32_t _pad2;
  /* optim */
  double  penalty_epsilon;
  double  weight_max_vel_x;
  double  weight_max_vel_y;
  double  weight_max_vel_theta;
  double  weight_acc_lim_x;
  double  weight_acc_lim_y;
  double  weight_acc_lim_theta;
  double  weight_kinematics_nh;
  double  weight_kinematics_forward_drive;
  double  weight_kinematics_turning_radius;
  double  weight_optimaltime;
  double  weight_shortest_path;
  double  weight_obstacle;
  double  weight_inflation;
  double  weight_dynamic_obstacle;
  double  weight_dynamic_obstacle_inflation;
  double  weight_velocity_obstacle_ratio;
  double  weight_viapoint;
  double  weight_prefer_rotdir;
  double  weight_adapt_factor;
  double  obstacle_cost_exponent;
  int32_t no_inner_iterations;
  int32_t no_outer_iterations;
  int32_t optimization_activate;
  int32_t _pad3;
  /* hcp (selection only) */
  double  selection_cost_hysteresis;
  double  selection_prefer_initial_plan;
  double  selection_obst_cost_scale;
  double  selection_viapoint_cost_scale;
  int32_t selection_alternative_time_cost;
  int32_t enable_multithreading;
  double  h_signature_prescaler;   /* teb_config.h:201, default 1   */
  double  h_signature_threshold;   /* teb_config.h:202, default 0.1 */
  /* recovery */
  int32_t divergence_detection_enable;
  int32_t _pad4;
  double  divergence_detection_max_chi_squared;
} TebParams;

/* Obstacle table row (64 bytes), constant-velocity model (obstacles.h:190-206).
 * Point / Circular (obstacles.h:305-445, :447-595): (x, y) is the position, radius the circle radius.
 * Line / Pill / Polygon (:597-740, :746-890, :893-1045): the shape is the vertex list
 * obst_vertices[scene][vertex_begin .. vertex_begin + vertex_count) (2 vertices for Line / Pill; a polygon is closed
 * implicitly when it has more than 2 vertices, distance_calculations.h:172-199), radius is the pill radius and (x, y)
 * must hold getCentroid() (line midpoint :734; polygon centroid obstacles.cpp:47-97) — the obstacle association uses
 * it to tell left from right (optimal_planner.cpp:503). */
typedef struct TebObstacle {
  double  x, y;          /* position / centroid */
  double  vx, vy;        /* centroid velocity (obstacles.h:206) */
  double  radius;        /* Circular, Pill; 0 otherwise */
  int32_t dynamic;       /* isDynamic() (obstacles.h:199) */
  int32_t type;          /* TEB_OBST_* */
  int32_t vertex_begin;  /* Line / Pill / Polygon: first vertex in the scene's vertex pool */
  int32_t vertex_count;
  double  _pad;
} TebObstacle;

/* A batch of bands (homotopy candidates x planning requests). All pointers are HOST pointers for
 * tebgpu_optimize_batch and DEVICE pointers for tebgpu_optimize_batch_device. */
typedef struct TebBatch {
  int32_t B;          /* number of bands                                   */
  int32_t n_cap;      /* records per band (stride); >= every n[b]           */
  int32_t S;          /* number of scenes (obstacle tables)                 */
  int32_t M_cap;      /* obstacle rows per scene (stride)                   */
  int32_t V_cap;      /* via-points per band (stride); may be 0             */
  int32_t PV_cap;     /* obstacle vertices per scene (stride); 0 <=> only Point / Circular obstacles */
  double*            poses;       /* [B][n_cap][4]  in/out                              */
  int32_t*           n;           /* [B]            in/out (autoResize changes it)      */
  const int32_t*     scene_id;    /* [B]                                                */
  const TebObstacle* obstacles;   /* [S][M_cap]                                         */
  const int32_t*     obst_count;  /* [S]                                                */
  const double*      obst_vertices; /* [S][PV_cap][2] vertex pool of the Line / Pill / Polygon obstacles, or NULL   */
  const double*      via;         /* [B][V_cap][2] or NULL                              */
  const int32_t*     via_count;   /* [B] or NULL                                        */
  const double*      vel_start;   /* [B][4] = vx, vy, omega, active(0/1)  (optimal_planner.cpp:233-245) */
  const double*      vel_goal;    /* [B][4] = vx, vy, omega, active(0/1); active=0 <=> free_goal_vel     */
  const int32_t*     prefer_rotdir; /* [B] TEB_ROTDIR_* or NULL (optimal_planner.cpp:961-997)           */
  double*            cost;        /* [B] out: getCurrentCost() (optimal_planner.h:437)  */
  double*            chi2;        /* [B] out: chi2 of the final state of the last LM iteration (hasDiverged) */
  int32_t*           status;      /* [B] out: TEB_STATUS_* bits                          */
  int32_t*           lm_iters;    /* [B] out: inner LM iterations executed (all outer iterations) */
} TebBatch;

/* Arguments of TebOptimalPlanner::optimizeTEB (optimal_planner.h:231). */
typedef struct TebOptimizeArgs {
  int32_t iterations_innerloop;
  int32_t iterations_outerloop;
  int32_t compute_cost_afterwards;
  int32_t alternative_time_cost;
  double  obst_cost_scale;
  double  viapoint_cost_scale;
} TebOptimizeArgs;

typedef struct TebGpuLimits {
  int32_t max_bands;      /* B capacity */
  int32_t max_poses;      /* n_cap capacity (<= 512) */
  int32_t max_scenes;
  int32_t max_obstacles;  /* M_cap capacity (<= 1024: 16 association words per pose; the scene's table is staged in shared memory) */
  int32_t max_viapoints;  /* V_cap capacity */
  int32_t max_obst_vertices; /* PV_cap capacity (0: Point / Circular obstacles only) */
} TebGpuLimits;

typedef struct tebgpu_ctx tebgpu_ctx;

/* Fill `p` with the TebConfig() constructor defaults (teb_config.h:245-390). The three fields the
 * reference leaves uninitialised in the ctor get their dynamic_reconfigure defaults
 * (divergence_detection_enable=0, divergence_detection_max_chi_squared=10). */
void tebgpu_default_params(TebParams* p);

/* sizeof() of the ABI structs, for binding sanity checks. which: 0 TebParams, 1 TebObstacle, 2 TebBatch,
 * 3 TebOptimizeArgs, 4 TebGpuLimits. */
int32_t tebgpu_sizeof(int32_t which);

/* Context life cycle. One context = one device + one stream + its device workspaces.
 * Replaces initOptimizer()/SparseOptimizer ownership (optimal_planner.cpp:161-179). */
int32_t tebgpu_create(const TebGpuLimits* limits, int32_t device, tebgpu_ctx** out);
int32_t tebgpu_destroy(tebgpu_ctx* ctx);
const char* tebgpu_last_error_string(const tebgpu_ctx* ctx);

/* cfg_ pointer equivalent (optimal_planner.h:675): parameters are copied, call again after changes. */
int32_t tebgpu_set_params(tebgpu_ctx* ctx, const TebParams* params);

/* optimizeTEB over a whole batch, HOST buffers: H2D copy, all outer x inner LM iterations on the
 * device, D2H copy of poses / n / cost / chi2 / status / lm_iters, synchronous.
 * Replaces HomotopyClassPlanner::optimizeAllTEBs' thread fan-out (homotopy_class_planner.cpp:466-493). */
int32_t tebgpu_optimize_batch(tebgpu_ctx* ctx, const TebBatch* batch, const TebOptimizeArgs* args);

/* Same, every pointer in `batch` is a DEVICE pointer on the context's device. Stream-ordered on the
 * context stream (or `cuda_stream` if non-NULL, a cudaStream_t passed as void*; NULL means the context's own
 * stream, so pass cudaStreamLegacy / cudaStreamPerThread explicitly to target a default stream); does NOT
 * synchronise. */
int32_t tebgpu_optimize_batch_device(tebgpu_ctx* ctx, const TebBatch* batch, const TebOptimizeArgs* args,
                                     void* cuda_stream);
int32_t tebgpu_synchronize(tebgpu_ctx* ctx);

/* Linear solver / scheduling of the LM step (replaces LinearSolverCSparse, optimal_planner.h:75-79):
 * 2 (default) speculative: the next 4 damping trials are solved concurrently, one thread per (band, trial), banded
 *   LDL^T with the active window in registers, and the accept / reject chain is replayed in order;
 * 1 block cyclic reduction on 8x8 blocks in shared memory (max_poses <= 256), one CTA per band;
 * 0 sequential banded LDL^T in shared memory, one CTA per band.  All three give the same results up to round-off. */
int32_t tebgpu_set_solver(tebgpu_ctx* ctx, int32_t solver);
/* Thread mapping of kernel A: 0 (default) k_linearize2: one thread per pose, 125-pose tiles, band rows accumulated in
 * registers; 1 the first-generation kernel: one 128-thread CTA per 32-pose tile, one thread per band row. Same
 * arithmetic, different summation order (results agree to round-off); variant 1 is kept as an independent cross-check. */
int32_t tebgpu_set_linearize_variant(tebgpu_ctx* ctx, int32_t variant);
/* Speculation width of solver 2: how many consecutive LM damping trials are solved per round (2, 4, 6 or 8; 0 = auto).
 * Results do not depend on it (the accept / reject chain is replayed in order), only latency and traffic do. */
int32_t tebgpu_set_speculation(tebgpu_ctx* ctx, int32_t k);

/* Mapping of the default solver's solve kernel (replaces LinearSolverCSparse::solve, optimal_planner.cpp:169-172):
 *   0  one THREAD per (band, trial) system (k_solve_tpb) always - the throughput mapping;
 *   1  one WARP per system (k_solve_warp: window spread over the lanes, pivot column through shared memory, axpy back
 *      substitution), 2 the same only while a round has at most 148 x 8 systems. Bit-identical to mode 0, measured 2.8x
 *      slower per solve on B200 (profiles/r2_history.md); kept as an independent cross-check of the factorisation;
 *   3  k_solve_lat always: one warp per system, the system resident in shared memory, TWISTED factorisation (the two
 *      half-warps eliminate from both ends towards an 11-unknown middle block), 2.6x faster per solve than mode 0 when
 *      the machine is not full; another elimination order, so results agree with mode 0 to rounding, not bit for bit;
 *   4  (default) k_solve_lat while the systems of a round fit three waves of resident CTAs - the latency regime of a
 *      single planning request - and k_solve_tpb above that. */
int32_t tebgpu_set_warp_solver(tebgpu_ctx* ctx, int32_t mode);

/* CUDA-graph replay of the launch sequence of tebgpu_optimize_batch(_device): 0 never, 1 always, 2 (default) in the
 * latency regime only (a batch of at most ~2300 bands, e.g. one planning request of 32 candidates, where the 130-170
 * kernel launches of one optimizeTEB are comparable to the kernels themselves). A sequence is captured once per distinct
 * (batch description incl. buffer addresses, optimize arguments, parameters, switches, stream) and replayed afterwards;
 * the context keeps the 8 most recently used graphs. Results are identical to direct launches. */
int32_t tebgpu_set_graph(tebgpu_ctx* ctx, int32_t mode);

/* Per-kernel device timing (CUDA events on the launching stream around every launch) for roofline reporting.
 * enable != 0 -> subsequent optimize calls record events. tebgpu_get_kernel_times synchronises, then returns for
 * kernel kind k (0 begin, 1 auto_resize, 2 build_graph, 3 linearize ["kernel A"], 4 lm_step [fused "kernel B" of
 * solvers 0/1; for solver 2: the solve/eval launches of the retry rounds >= 1], 5 finalize, 6 solve_tpb round 0,
 * 7 trial_eval round 0 (includes the accept / reject replay), 8 unused since the replay was fused into trial_eval
 * ["kernel B" of the default speculative solver])
 * the accumulated milliseconds and launch count since profiling was enabled, and resets the accumulators. */
int32_t tebgpu_set_profiling(tebgpu_ctx* ctx, int32_t enable);
int32_t tebgpu_get_kernel_times(tebgpu_ctx* ctx, double ms_out[9], int64_t count_out[9]);

/* HomotopyClassPlanner::calculateEquivalenceClass (homotopy_class_planner.hpp:46-63) for every band of the batch, i.e.
 * the step that decides which candidates are kept before they are optimised (renewAndAnalyzeOldTebs,
 * homotopy_class_planner.cpp:214-256). include_dynamic_obstacles == 0: HSignature (h_signature.h:97-186), h_out[b] =
 * (Re H, Im H), stride 2; otherwise HSignature3d (h_signature.h:282-353), h_out[b][l] for the M obstacles of the band's
 * scene, stride M_cap. The path is the band's pose positions; use_timediffs != 0 takes the transition times from the
 * band's dt, 0 approximates them by |z2 - z1| / max_vel_x (h_signature.h:307-315, graph-search candidates have no time
 * information yet). The reference accumulates the 2-D signature in long double; the device uses fp64 (|dH| <= 1e-9 |H|
 * against the long double oracle, far below h_signature_threshold). device_ptrs as in tebgpu_build_system. */
int32_t tebgpu_h_signature(tebgpu_ctx* ctx, const TebBatch* batch, int32_t use_timediffs, double* h_out, int32_t device_ptrs);

/* Number of kernels launched by the last optimize call (for bench.py's gpu_launches). */
int64_t tebgpu_last_launch_count(const tebgpu_ctx* ctx);
/* Introspection for measurement scripts. which: 0 speculation width used by the last optimize call, 1 kernel-A variant,
 * 2 solver, 3 communicator size (1 without tebgpu_comm_init), 4 communicator rank, 5 CUDA-graph replay enabled,
 * 6 number of captured graphs held by the context, 7 speculation width of the first LM iteration after a graph rebuild
 * (key 0 reports the width of the later iterations). Returns -1 for an unknown key. */
int64_t tebgpu_get_info(const tebgpu_ctx* ctx, int32_t which);

/* Linearise only: build the padded banded normal equations of every band at its current state for
 * outer iteration `outer_index` (obstacle weight multiplier = weight_adapt_factor^outer_index).
 * Hb_out [B][4*n_cap][12] (device or host per `device_ptrs`): row r = 11 lower-band entries
 * H[r][r-k], k=0..10, then b[r]; chi2_out[B]. Test / profiling entry point for kernel A
 * (BlockSolver::buildSystem, SURVEY §3.3 step 2). */
int32_t tebgpu_build_system(tebgpu_ctx* ctx, const TebBatch* batch, int32_t outer_index,
                            double* Hb_out, double* chi2_out, int32_t device_ptrs);

/* LM linear solve only (test entry point for the solve kernels of the default solver): for every band b and trial
 * k < K (1 .. 8), solve (H_b + lambda_bk * I_real) dx = b_b with the mapping chosen by tebgpu_set_warp_solver (0 thread,
 * 1 warp, 3 twisted; 2 and 4 resolve by the number of systems B * K as in optimize), where lambda_bk is lambda[b]
 * escalated k times (lambda *= ni, ni *= 2), as the speculative rounds do. I_real is the identity on the real unknowns:
 * rows 0 .. 2 (start pose) and 4 n - 4 .. 4 n - 1 (goal pose, dt of the last pose) are identity rows of H.
 * Same grid, shared memory and kernel choice as round 0 of an LM iteration of tebgpu_optimize_batch.
 * HOST buffers: Hb [B][4 n_cap][12] in the layout tebgpu_build_system writes, n [B] (3 .. n_cap), lambda [B], ni [B];
 * outputs dx_out [B][K][4 n_cap] (rows a kernel does not write - 4 n[b] .. 4 n_cap - 1, and the whole system after a
 * failed factorisation in modes 0 / 1 - are NaN), ok_out [B][K] (1: the factorisation succeeded, the flag the trial
 * evaluation reads; 0: TEB_STATUS_CHOL_FAILED), lambda_out [B][K] (the damping the kernel used). */
int32_t tebgpu_solve_system(tebgpu_ctx* ctx, int32_t B, int32_t n_cap, const int32_t* n, const double* Hb,
                            const double* lambda, const double* ni, int32_t K,
                            double* dx_out, int32_t* ok_out, double* lambda_out);

/* TebOptimalPlanner::computeCurrentCost called OUTSIDE optimizeTEB (optimal_planner.cpp:1041-1094, graph rebuilt with
 * weight multiplier 1, errors evaluated at the current state): HOST buffers; writes cost[], chi2[], status[]. */
int32_t tebgpu_compute_cost(tebgpu_ctx* ctx, const TebBatch* batch, const TebOptimizeArgs* args);

/* HomotopyClassPlanner::selectBestTeb (homotopy_class_planner.cpp:564-667) on gathered costs:
 * argmin over cost[i], with cost[last_best] * selection_cost_hysteresis and
 * cost[initial_plan] * selection_prefer_initial_plan (pass -1 for none). Strict '<', first wins.
 * Host-side, pure function. Returns the index or -1 if count == 0. */
int32_t tebgpu_select_best(const double* cost, int32_t count, int32_t last_best, int32_t initial_plan,
                           double selection_cost_hysteresis, double selection_prefer_initial_plan);

/* ---- multi-GPU: one process (or thread) per GPU, each with its own context; the batch axis is sharded and bands never
 * exchange anything while they are optimised. What replaces the join of HomotopyClassPlanner::optimizeAllTEBs' thread
 * fan-out (homotopy_class_planner.cpp:466-493) before selectBestTeb (:564-616) is ONE all-gather of the per-candidate
 * costs over NCCL on the context's stream. NCCL is resolved at run time (dlopen); single-GPU users never load it.
 *   tebgpu_comm_get_unique_id  rank 0 creates the 128-byte id and distributes it out of band (MPI, a store, a file)
 *   tebgpu_comm_init           every rank, collectively: ncclCommInitRank on the context's device
 *   tebgpu_gather_costs        cost_all[r * count_local + k] = cost_local of rank r (same count on every rank);
 *                              device_ptrs != 0: both pointers are device memory, stream ordered on `cuda_stream` (a
 *                              cudaStream_t as void*; NULL = the context's stream, as in tebgpu_optimize_batch_device), no
 *                              synchronisation; 0: host memory, synchronous. Without a communicator (one rank): a copy.
 *   tebgpu_optimize_batch_gather  tebgpu_optimize_batch followed by the gather of batch->cost: cost_all [world * B] (host)
 * Errors: TEBGPU_ERR_UNSUPPORTED when NCCL cannot be loaded, TEBGPU_ERR_CUDA for NCCL / CUDA failures (see
 * tebgpu_last_error_string). */
#define TEBGPU_COMM_ID_BYTES 128
int32_t tebgpu_comm_get_unique_id(void* id_out);
int32_t tebgpu_comm_init(tebgpu_ctx* ctx, const void* id, int32_t world_size, int32_t rank);
int32_t tebgpu_comm_destroy(tebgpu_ctx* ctx);
int32_t tebgpu_gather_costs(tebgpu_ctx* ctx, const double* cost_local, int32_t count_local, double* cost_all, int32_t device_ptrs,
                            void* cuda_stream);
int32_t tebgpu_optimize_batch_gather(tebgpu_ctx* ctx, const TebBatch* batch, const TebOptimizeArgs* args, double* cost_all);

/* TimedElasticBand::autoResize (timed_elastic_band.cpp:227-286) on one host band; same routine the
 * device kernel runs. rec: [n_cap][4] in/out, returns the new n (or <0 on error). */
int32_t tebgpu_auto_resize_host(double* rec, int32_t n, int32_t n_cap, double dt_ref, double dt_hysteresis,
                                int32_t min_samples, int32_t max_samples, int32_t fast_mode);

#ifdef __cplusplus
}
#endif
#endif /* TEB_B200_H */
