/*
 * teb_cabi.cu — C-ABI (include/teb_b200.h) over the sm_100a kernels in teb_kernels.cuh.
 * No CPU fallback: every entry point that optimises needs a CUDA device and fails loudly otherwise.
 */
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "teb_kernels.cuh"
#include "teb_linearize.cuh"
#include "teb_spec.cuh"
#include "teb_solve_warp.cuh"
#include "teb_solve_lat.cuh"
#include "teb_hsig.cuh"
#include "teb_comm.h"
#include <cstdlib>

using namespace tebgpu;

struct tebgpu_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;        /* retry rounds of the speculative solver, overlapped with the next kernel A */
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_s0 = nullptr;
  double* Lf2 = nullptr;              /* scratch of the side stream's solver launches (they overlap the main stream's) */
  double* dx2 = nullptr;
  int split = 1;                      /* throughput regime: the side stream also runs round 0 for its bands (TEBGPU_SPLIT) */
  int overlap = 2;                    /* retry rounds on the side stream: 0 never (one stream), 1 always, 2 (default) only in the
                                         latency regime - measured on C2 / C3 / C4 at 8192 bands the three schedules are within
                                         +-3 % of each other, the machine is resource bound there (TEBGPU_OVERLAP) */
  int32_t* defer = nullptr;           /* [B] */
  double* d_fp = nullptr;             /* footprint definition for the vertex-list distance path (FP_DOUBLES) */
  double* d_pverts = nullptr;         /* [S][max_obst_vertices][2] mirror of TebBatch.obst_vertices */
  double* d_hsig = nullptr;           /* [max_bands][max(max_obstacles, 2)] H-signature output of the host-buffer entry point */
  TebGpuLimits lim{};
  TebParams params{};
  bool have_params = false;
  std::string err;
  int64_t launches = 0;
  int linearize_variant = 0;  /* 0: k_linearize2, one thread per pose, 125-pose tiles (default);
                                 1: k_linearize, first generation: 128-thread CTA per 32-pose tile, thread per band row */
  ncclComm_t comm = nullptr;          /* cost all-gather across the ranks of a sharded batch (tebgpu_comm_init) */
  int world = 1, rank = 0;
  int32_t* arrive = nullptr;          /* [max_bands] k_trial_eval3: CTAs of a band that have published their trial (0 between rounds) */
  int eval_mode = 2;                  /* 2 automatic (k_trial_eval3 in the latency regime), 0 k_trial_eval2 always, 1 k_trial_eval3 always (TEBGPU_EVAL3) */
  double* d_gather = nullptr;         /* [world][max_bands] gathered costs of the host-buffer entry point */
  struct GraphEntry { uint64_t key = 0; cudaGraphExec_t exec = nullptr; int64_t launches = 0; uint64_t stamp = 0; int spec_k = 0, spec_first = 0; };
  std::vector<GraphEntry> graphs;     /* captured launch sequences (tebgpu_set_graph) */
  uint64_t graph_clock = 0;
  uint64_t params_version = 0;        /* bumped by tebgpu_set_params: part of the graph key */
  int graph_mode = 2;                 /* 0 never, 1 always, 2 automatic (latency regime only) */
  int warp_solver = 4; /* solver 2, solve kernel (TEBGPU_WARP_SOLVER / tebgpu_set_warp_solver):
                          0 thread per system (k_solve_tpb) always,
                          1 / 2 k_solve_warp always / in the latency regime - measured 2.8x SLOWER per solve than k_solve_tpb,
                            kept as an independently mapped, bit-identical implementation,
                          3 / 4 k_solve_lat (twisted factorisation, system resident in shared memory) always / while the
                            systems of a round fit LAT_WAVES waves of resident CTAs (the latency regime; DEFAULT) */
  int ring = 0;        /* solver prefetch ring: 0 = 10 rows (default), else 10 / 20 / 30 rows (TEBGPU_RING, experiments) */
  int eval_v1 = 0;     /* TEBGPU_EVAL_V1=1: first-generation trial evaluation (warp per trial, chunk per lane) */
  int ka_staged = 1;   /* kernel A output: 1 (default) shared-memory slot + TMA bulk store per lane, 0 direct 128-bit global stores */
  int last_spec_k = 0; /* round-0 width of the later LM iterations of the last optimize call */
  int last_spec_first = 0; /* round-0 width of the first LM iteration after a graph rebuild */
  int spec_k = 0;  /* speculation width: 0 = auto (6 when B*6 systems fit one warp per SM sub-partition, else 4) */
  int solver = 2;  /* 2: speculative thread-per-(band,trial) LDL^T (default), 1: block cyclic reduction, 0: sequential */
  int MW = 1;
  int chunks = 1;
  /* device workspaces */
  double* Hb = nullptr;
  unsigned long long* assoc = nullptr;
  unsigned long long* assoc3 = nullptr;
  double* dyn_t = nullptr;
  int32_t* via_idx = nullptr;
  double* chi_parts = nullptr;
  double* dmax_parts = nullptr;
  double* rhs = nullptr;
  int32_t* dyn_idx = nullptr;
  int32_t* dyn_cnt = nullptr;
  SpecBufs spec{};
  int eval_minb = 3; /* k_trial_eval register budget: 3 -> 80 registers, 6 CTAs/SM (measured 3-4 % faster than 2 -> 122
                        registers, 4 CTAs/SM, despite 180 bytes of spills); TEBGPU_EVAL_MINB=2 selects the other build */
  BandState* state = nullptr;
  /* device mirrors for the host-buffer entry point */
  double* d_poses = nullptr; int32_t* d_n = nullptr; int32_t* d_scene = nullptr; TebObstacle* d_obst = nullptr;
  int32_t* d_ocount = nullptr; double* d_via = nullptr; int32_t* d_vcount = nullptr; double* d_vs = nullptr;
  double* d_vg = nullptr; int32_t* d_rot = nullptr; double* d_cost = nullptr; double* d_chi2 = nullptr;
  int32_t* d_status = nullptr; int32_t* d_iters = nullptr;
  size_t smem_a = 0, smem_b = 0, smem_g = 0;
  /* profiling */
  bool profiling = false;
  std::vector<cudaEvent_t> ev;      /* pairs */
  std::vector<int> ev_kind;
  size_t ev_used = 0;
  double prof_ms[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int64_t prof_cnt[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
};

static void prof_begin(tebgpu_ctx* c, cudaStream_t st, int kind) {
  if (!c->profiling) return;
  if (c->ev_used + 2 > c->ev.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    c->ev.push_back(a);
    c->ev.push_back(b);
    c->ev_kind.push_back(kind);
  }
  c->ev_kind[c->ev_used / 2] = kind;
  cudaEventRecord(c->ev[c->ev_used], st);
}
static void prof_end(tebgpu_ctx* c, cudaStream_t st) {
  if (!c->profiling) return;
  cudaEventRecord(c->ev[c->ev_used + 1], st);
  c->ev_used += 2;
}
static void prof_collect(tebgpu_ctx* c) {
  for (size_t k = 0; k + 1 < c->ev_used + 1 && k < c->ev_used; k += 2) {
    float ms = 0;
    cudaEventSynchronize(c->ev[k + 1]);
    cudaEventElapsedTime(&ms, c->ev[k], c->ev[k + 1]);
    c->prof_ms[c->ev_kind[k / 2]] += ms;
    c->prof_cnt[c->ev_kind[k / 2]] += 1;
  }
  c->ev_used = 0;
}

#define CUDA_TRY(ctx, expr)                                                                      \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                           \
      return TEBGPU_ERR_CUDA;                                                                    \
    }                                                                                            \
  } while (0)

extern "C" {

void tebgpu_default_params(TebParams* p) {
  /* TebConfig::TebConfig() teb_config.h:245-390 */
  std::memset(p, 0, sizeof(*p));
  p->dt_ref = 0.3; p->dt_hysteresis = 0.1;
  p->force_reinit_new_goal_dist = 1; p->force_reinit_new_goal_angular = 0.5 * M_PI;
  p->teb_autosize = 1; p->min_samples = 3; p->max_samples = 500; p->exact_arc_length = 0;
  p->via_points_ordered = 0; p->allow_init_with_backwards_motion = 0; p->global_plan_overwrite_orientation = 1;
  p->max_vel_x = 0.4; p->max_vel_x_backwards = 0.2; p->max_vel_y = 0.0; p->max_vel_trans = 0.0; p->max_vel_theta = 0.3;
  p->acc_lim_x = 0.5; p->acc_lim_y = 0.5; p->acc_lim_theta = 0.5; p->min_turning_radius = 0;
  p->footprint_type = TEB_FOOTPRINT_POINT;
  p->min_obstacle_dist = 0.5; p->inflation_dist = 0.6; p->dynamic_obstacle_inflation_dist = 0.6;
  p->obstacle_association_force_inclusion_factor = 1.5; p->obstacle_association_cutoff_factor = 5;
  p->obstacle_proximity_ratio_max_vel = 1; p->obstacle_proximity_lower_bound = 0; p->obstacle_proximity_upper_bound = 0.5;
  p->include_dynamic_obstacles = 1; p->legacy_obstacle_association = 0; p->obstacle_poses_affected = 25;
  p->penalty_epsilon = 0.05;
  p->weight_max_vel_x = 2; p->weight_max_vel_y = 2; p->weight_max_vel_theta = 1;
  p->weight_acc_lim_x = 1; p->weight_acc_lim_y = 1; p->weight_acc_lim_theta = 1;
  p->weight_kinematics_nh = 1000; p->weight_kinematics_forward_drive = 1; p->weight_kinematics_turning_radius = 1;
  p->weight_optimaltime = 1; p->weight_shortest_path = 0;
  p->weight_obstacle = 50; p->weight_inflation = 0.1;
  p->weight_dynamic_obstacle = 50; p->weight_dynamic_obstacle_inflation = 0.1;
  p->weight_velocity_obstacle_ratio = 0; p->weight_viapoint = 1; p->weight_prefer_rotdir = 50;
  p->weight_adapt_factor = 2.0; p->obstacle_cost_exponent = 1.0;
  p->no_inner_iterations = 5; p->no_outer_iterations = 4; p->optimization_activate = 1;
  p->selection_cost_hysteresis = 1.0; p->selection_prefer_initial_plan = 0.95;
  p->selection_obst_cost_scale = 100.0; p->selection_viapoint_cost_scale = 1.0;
  p->selection_alternative_time_cost = 0; p->enable_multithreading = 1;
  p->h_signature_prescaler = 1; p->h_signature_threshold = 0.1;
  p->divergence_detection_enable = 0; p->divergence_detection_max_chi_squared = 10;
}

int32_t tebgpu_sizeof(int32_t which) {
  switch (which) {
    case 0: return (int32_t)sizeof(TebParams);
    case 1: return (int32_t)sizeof(TebObstacle);
    case 2: return (int32_t)sizeof(TebBatch);
    case 3: return (int32_t)sizeof(TebOptimizeArgs);
    case 4: return (int32_t)sizeof(TebGpuLimits);
    default: return -1;
  }
}

const char* tebgpu_last_error_string(const tebgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
int64_t tebgpu_last_launch_count(const tebgpu_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t tebgpu_get_info(const tebgpu_ctx* ctx, int32_t which) {
  if (!ctx) return -1;
  switch (which) {
    case 0: return ctx->last_spec_k;
    case 1: return ctx->linearize_variant;
    case 2: return ctx->solver;
    case 3: return ctx->world;
    case 4: return ctx->rank;
    case 5: return ctx->graph_mode;
    case 6: return (int64_t)ctx->graphs.size();
    case 7: return ctx->last_spec_first;
    default: return -1;
  }
}

static void free_all(tebgpu_ctx* c) {
  void* ptrs[] = {c->Lf2, c->dx2, c->arrive, c->d_gather, c->d_hsig, c->assoc3, c->dyn_idx, c->dyn_cnt, c->rhs, c->dmax_parts, c->spec.Lf, c->spec.dx, c->spec.res, c->spec.need, c->spec.qmax, c->spec.cnt, c->spec.list, c->defer, c->d_fp, c->d_pverts, c->Hb, c->assoc, c->dyn_t, c->via_idx, c->chi_parts, c->state, c->d_poses, c->d_n, c->d_scene,
                  c->d_obst, c->d_ocount, c->d_via, c->d_vcount, c->d_vs, c->d_vg, c->d_rot, c->d_cost, c->d_chi2,
                  c->d_status, c->d_iters};
  for (void* p : ptrs)
    if (p) cudaFree(p);
}

int32_t tebgpu_create(const TebGpuLimits* lim, int32_t device, tebgpu_ctx** out) {
  if (!lim || !out) return TEBGPU_ERR_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= device || device < 0) {
    std::fprintf(stderr, "tebgpu_create: no CUDA device %d available (this library has no CPU fallback)\n", device);
    return TEBGPU_ERR_NO_DEVICE;
  }
  if (lim->max_bands < 1 || lim->max_poses < 3 || lim->max_poses > 512 || lim->max_scenes < 1 || lim->max_obstacles < 0 ||
      lim->max_obstacles > 64 * MAX_MW || lim->max_viapoints < 0 || lim->max_obst_vertices < 0)
    return TEBGPU_ERR_INVALID_ARG;
  tebgpu_ctx* c = new (std::nothrow) tebgpu_ctx();
  if (!c) return TEBGPU_ERR_CUDA;
  c->device = device;
  c->lim = *lim;
  if (c->lim.max_obstacles < 1) c->lim.max_obstacles = 1;
  c->MW = (c->lim.max_obstacles + 63) / 64;
  c->chunks = (c->lim.max_poses + KA2_TP - 1) / KA2_TP; /* capacity for the smaller of the two tile sizes */
  *out = c;
  CUDA_TRY(c, cudaSetDevice(device));
  CUDA_TRY(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  {
    int lo = 0, hi = 0; /* the latency-bound retry chain should never queue behind the bulk kernels */
    CUDA_TRY(c, cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CUDA_TRY(c, cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, hi));
  }
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
  CUDA_TRY(c, cudaEventCreateWithFlags(&c->ev_s0, cudaEventDisableTiming));
  if (const char* e = std::getenv("TEBGPU_OVERLAP")) { const int m = std::atoi(e); if (m >= 0 && m <= 2) c->overlap = m; }
  if (const char* e = std::getenv("TEBGPU_SPEC_K")) { const int k = std::atoi(e); if (k == 2 || k == 4 || k == 6 || k == 8) c->spec_k = k; }
  const size_t B = c->lim.max_bands, nc = c->lim.max_poses, S = c->lim.max_scenes, M = c->lim.max_obstacles,
               V = c->lim.max_viapoints > 0 ? c->lim.max_viapoints : 1;
  CUDA_TRY(c, cudaMalloc(&c->Hb, B * 4 * nc * HROW * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->assoc, B * nc * c->MW * sizeof(unsigned long long)));
  CUDA_TRY(c, cudaMalloc(&c->assoc3, B * nc * c->MW * sizeof(unsigned long long)));
  CUDA_TRY(c, cudaMalloc(&c->dyn_t, B * nc * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->via_idx, B * V * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->chi_parts, B * c->chunks * 4 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->state, B * sizeof(BandState)));
  CUDA_TRY(c, cudaMalloc(&c->dmax_parts, B * c->chunks * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->rhs, B * 4 * nc * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->dyn_idx, S * M * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->dyn_cnt, S * sizeof(int32_t)));
  {
    size_t ev = eval_smem_bytes((int)nc, (int)M, SPEC_K_MAX);
    if (ev > 232448) ev = 232448; /* wide speculation is only chosen when its staging fits (tebgpu_optimize_batch_device) */
    CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev));
    CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev));
    CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev));
    if (const char* e = std::getenv("TEBGPU_EVAL3")) { const int m = std::atoi(e); if (m >= 0 && m <= 2) c->eval_mode = m; }
    if (const char* e = std::getenv("TEBGPU_EVAL_MINB")) c->eval_minb = std::atoi(e) == 3 ? 3 : 2;
    if (const char* e = std::getenv("TEBGPU_EVAL_V1")) c->eval_v1 = std::atoi(e) != 0;
    size_t ev2 = eval2_smem_bytes((int)nc, (int)M, SPEC_K_MAX);
    if (ev2 > 232448) ev2 = 232448;
#define EV2_ATTR(G, T)                                                                                                  \
  CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval2<G, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev2));          \
  CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval2<G, T>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    EV2_ATTR(false, 256) EV2_ATTR(true, 256) EV2_ATTR(false, 512) EV2_ATTR(true, 512)
#undef EV2_ATTR
    size_t ev3 = eval3_smem_bytes((int)nc, (int)M, SPEC_K_MAX);
    if (ev3 > 232448) ev3 = 232448;
    CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev3));
    CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ev3));
  }
  const size_t spec_sys = ((B * SPEC_K_MAX + 31) / 32) * 32; /* whole warps of (band, trial) systems */
  CUDA_TRY(c, cudaMalloc(&c->spec.Lf, spec_sys * 4 * nc * HROW * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->spec.dx, spec_sys * 4 * nc * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->Lf2, spec_sys * 4 * nc * HROW * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->dx2, spec_sys * 4 * nc * sizeof(double)));
  c->spec.sel_list = nullptr; c->spec.sel_cnt = nullptr; c->spec.defer = nullptr; c->spec.skip_tag = 0; c->spec.lat_cap = 0;
  if (const char* e = std::getenv("TEBGPU_SPLIT")) c->split = std::atoi(e) != 0;
  CUDA_TRY(c, cudaMalloc(&c->spec.cnt, SPEC_CNT_CAP * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->spec.list, SPEC_LISTS * B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->defer, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->spec.res, B * SPEC_K_MAX * RES_STRIDE * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->arrive, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMemset(c->arrive, 0, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->spec.need, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->spec.qmax, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_poses, B * nc * 4 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_n, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_scene, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_obst, S * M * sizeof(TebObstacle)));
  CUDA_TRY(c, cudaMalloc(&c->d_ocount, S * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_via, B * V * 2 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_fp, FP_DOUBLES * sizeof(double)));
  CUDA_TRY(c, cudaMemset(c->d_fp, 0, FP_DOUBLES * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_pverts, (S * (size_t)(lim->max_obst_vertices > 0 ? lim->max_obst_vertices : 1)) * 2 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_hsig, B * (M > 2 ? M : 2) * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_vcount, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_vs, B * 4 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_vg, B * 4 * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_rot, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_cost, B * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_chi2, B * sizeof(double)));
  CUDA_TRY(c, cudaMalloc(&c->d_status, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMalloc(&c->d_iters, B * sizeof(int32_t)));
  CUDA_TRY(c, cudaMemsetAsync(c->dyn_t, 0, B * nc * sizeof(double), c->stream));
  CUDA_TRY(c, cudaMemsetAsync(c->via_idx, 0xff, B * V * sizeof(int32_t), c->stream));
  c->smem_a = ka_smem_bytes((int)M);
  c->smem_b = kb_smem_bytes((int)nc, (int)M);
  c->smem_g = M * sizeof(TebObstacle);
  if (c->smem_b > 232448 || c->smem_a > 232448) {
    c->err = "shared-memory footprint exceeds 227 KB for these limits (max_poses / max_obstacles too large)";
    return TEBGPU_ERR_CAPACITY;
  }
  if (ka2_smem_bytes<true>((int)M) > 232448) {
    c->err = "kernel A staging exceeds 227 KB for these limits (max_obstacles too large)";
    return TEBGPU_ERR_CAPACITY;
  }
#define KA2_ATTR(H, G, O)                                                                                                    \
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize2<H, G, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ka2_smem_bytes<H>((int)M))); \
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize2<H, G, O>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  KA2_ATTR(false, false, true) KA2_ATTR(false, true, true) KA2_ATTR(true, false, true) KA2_ATTR(true, true, true)
  KA2_ATTR(false, false, false) KA2_ATTR(false, true, false) KA2_ATTR(true, false, false) KA2_ATTR(true, true, false)
#undef KA2_ATTR
  c->ka_staged = 1; /* measured: 0.44 ms (TMA bulk store per lane) vs 0.55 ms (direct 128-bit stores) per launch at C3 */
  if (const char* e = std::getenv("TEBGPU_KA_STAGED")) c->ka_staged = std::atoi(e) != 0;
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_a));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_a));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_a));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_a));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<0, KB_THREADS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_b));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<0, KB_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_b));
  if ((int)nc <= BCR_MAX_POSES && kb_bcr_smem_bytes((int)nc, (int)M) <= 232448) {
    CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<1, KB_BCR_THREADS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kb_bcr_smem_bytes((int)nc, (int)M)));
    CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<1, KB_BCR_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kb_bcr_smem_bytes((int)nc, (int)M)));
  }
  CUDA_TRY(c, cudaFuncSetAttribute(k_build_graph<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_g));
  CUDA_TRY(c, cudaFuncSetAttribute(k_build_graph<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_g));
  /* ask for the full shared-memory carveout: occupancy of the tile kernels is shared-memory bound */
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_linearize<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_tpb<10>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_tpb<20>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_tpb<30>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_tpb<20>, cudaFuncAttributeMaxDynamicSharedMemorySize, tpb_ring_bytes(20)));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_tpb<30>, cudaFuncAttributeMaxDynamicSharedMemorySize, tpb_ring_bytes(30)));
  CUDA_TRY(c, cudaFuncSetAttribute(k_solve_lat, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
  if (const char* e = std::getenv("TEBGPU_LAT_TIMING")) { const int v = std::atoi(e); CUDA_TRY(c, cudaMemcpyToSymbol(g_lat_timing, &v, sizeof(int))); }
  if (const char* e = std::getenv("TEBGPU_WARP_SOLVER")) { const int m = std::atoi(e); if (m >= 0 && m <= 4) c->warp_solver = m; }
  if (const char* e = std::getenv("TEBGPU_GRAPH")) { const int m = std::atoi(e); if (m >= 0 && m <= 2) c->graph_mode = m; }
  if (const char* e = std::getenv("TEBGPU_RING")) { const int r = std::atoi(e); if (r == 10 || r == 20 || r == 30) c->ring = r; }
  CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<2, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<2, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_trial_eval<3, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<0, KB_THREADS, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<0, KB_THREADS, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<1, KB_BCR_THREADS, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  CUDA_TRY(c, cudaFuncSetAttribute(k_lm_step_t<1, KB_BCR_THREADS, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  tebgpu_default_params(&c->params);
  c->have_params = true;
  CUDA_TRY(c, cudaStreamSynchronize(c->stream));
  return TEBGPU_OK;
}

int32_t tebgpu_destroy(tebgpu_ctx* ctx) {
  if (!ctx) return TEBGPU_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->stream) { cudaStreamSynchronize(ctx->stream); }
  if (ctx->comm) { nccl_api().CommDestroy(ctx->comm); ctx->comm = nullptr; }
  for (auto& e : ctx->graphs) cudaGraphExecDestroy(e.exec);
  ctx->graphs.clear();
  free_all(ctx);
  for (cudaEvent_t e : ctx->ev) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->side) cudaStreamDestroy(ctx->side);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->ev_s0) cudaEventDestroy(ctx->ev_s0);
  delete ctx;
  return TEBGPU_OK;
}

int32_t tebgpu_set_params(tebgpu_ctx* ctx, const TebParams* p) {
  if (!ctx || !p) return TEBGPU_ERR_INVALID_ARG;
  if (p->footprint_type < 0 || p->footprint_type > TEB_FOOTPRINT_POLYGON) { ctx->err = "unknown footprint model"; return TEBGPU_ERR_UNSUPPORTED; }
  if (p->footprint_type == TEB_FOOTPRINT_POLYGON &&
      (p->footprint_vertex_count < 1 || p->footprint_vertex_count > TEB_MAX_FOOTPRINT_VERTICES)) {
    ctx->err = "polygon footprint needs 1 .. TEB_MAX_FOOTPRINT_VERTICES vertices";
    return TEBGPU_ERR_INVALID_ARG;
  }
  /* footprint definition for the vertex-list distance path: a small device array, read by generic_distance */
  double fp[FP_DOUBLES];
  std::memset(fp, 0, sizeof(fp));
  fp[FP_RADIUS] = p->footprint_radius;
  fp[FP_FRONT_OFF] = p->footprint_front_offset; fp[FP_FRONT_RAD] = p->footprint_front_radius;
  fp[FP_REAR_OFF] = p->footprint_rear_offset; fp[FP_REAR_RAD] = p->footprint_rear_radius;
  for (int k = 0; k < 4; ++k) fp[FP_LINE + k] = p->footprint_line[k];
  fp[FP_COUNT] = (double)p->footprint_vertex_count;
  for (int k = 0; k < 2 * TEB_MAX_FOOTPRINT_VERTICES; ++k) fp[FP_VERTS + k] = p->footprint_vertices[k];
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream)); /* no optimize call of this context may still read the old copy */
  CUDA_TRY(ctx, cudaMemcpy(ctx->d_fp, fp, sizeof(fp), cudaMemcpyHostToDevice));
  ctx->params = *p;
  ctx->have_params = true;
  ++ctx->params_version;
  return TEBGPU_OK;
}

/* Kernel instantiations: HOLO = holonomic rows (vy, acc y); GEOM = vertex-list shapes (Line / Polygon footprint,
 * Line / Pill / Polygon obstacles) reachable, i.e. the out-of-line generic_distance call is compiled in. The default
 * diff-drive / car-like + Point / Circular configuration runs <false, false>: no extra rows, no call. */
static void launch_linearize(tebgpu_ctx* ctx, const DevBatch& db, const KParams& kp, int B, int M_cap, cudaStream_t st) {
  const bool holo = kp.holo_vel || kp.holo_acc;
  const bool geom = kp.generic != 0;
  if (ctx->linearize_variant == 1) {
    const dim3 grid(db.chunks, B);
    const size_t sm = ka_smem_bytes(M_cap);
    if (holo && geom) k_linearize<true, true><<<grid, KA_THREADS, sm, st>>>(db, kp);
    else if (holo) k_linearize<true, false><<<grid, KA_THREADS, sm, st>>>(db, kp);
    else if (geom) k_linearize<false, true><<<grid, KA_THREADS, sm, st>>>(db, kp);
    else k_linearize<false, false><<<grid, KA_THREADS, sm, st>>>(db, kp);
  } else {
    const dim3 g2((db.chunks + KA2_W - 1) / KA2_W, B);
    const size_t sm = holo ? ka2_smem_bytes<true>(M_cap) : ka2_smem_bytes<false>(M_cap);
#define KA2_LAUNCH(H, G)                                                                      \
  do {                                                                                        \
    if (ctx->ka_staged) k_linearize2<H, G, false><<<g2, KA2_THREADS, sm, st>>>(db, kp);       \
    else k_linearize2<H, G, true><<<g2, KA2_THREADS, sm, st>>>(db, kp);                       \
  } while (0)
    if (holo && geom) KA2_LAUNCH(true, true);
    else if (holo) KA2_LAUNCH(true, false);
    else if (geom) KA2_LAUNCH(false, true);
    else KA2_LAUNCH(false, false);
#undef KA2_LAUNCH
  }
}
static void launch_build_graph(const DevBatch& db, const KParams& kp, int B, size_t smem, cudaStream_t st) {
  if (kp.generic) k_build_graph<true><<<B, 256, smem, st>>>(db, kp);
  else k_build_graph<false><<<B, 256, smem, st>>>(db, kp);
}
static void launch_vor(const DevBatch& db, const KParams& kp, int B, size_t smem, cudaStream_t st) {
  if (kp.generic) k_vor<true><<<B, 256, smem, st>>>(db, kp);
  else k_vor<false><<<B, 256, smem, st>>>(db, kp);
}
static size_t eval_bytes(const tebgpu_ctx* ctx, int n_cap, int M_cap, int K) {
  return ctx->eval_v1 ? eval_smem_bytes(n_cap, M_cap, K) : eval2_smem_bytes(n_cap, M_cap, K);
}
static void launch_trial_eval(tebgpu_ctx* ctx, const SpecBufs& spec, const DevBatch& db, const KParams& kp, int B, int K,
                              size_t smem, int it, int round, int g, int tag, cudaStream_t st) {
  /* latency regime: a CTA per (band, trial) instead of a CTA per band while that still fits ~3 CTAs per SM */
  const size_t smem3 = eval3_smem_bytes(db.n_cap, db.M_cap, K);
  if (!ctx->eval_v1 && smem3 <= 232448 && (ctx->eval_mode == 1 || (ctx->eval_mode == 2 && (long long)B * K <= 148 * 3))) {
    int warps = ev2_tiles(db.n_cap);
    warps = warps < 1 ? 1 : (warps > 16 ? 16 : warps);
    const dim3 grid(K, B);
    if (kp.generic) k_trial_eval3<true><<<grid, 32 * warps, smem3, st>>>(db, kp, spec, it, round, g, tag, ctx->arrive);
    else k_trial_eval3<false><<<grid, 32 * warps, smem3, st>>>(db, kp, spec, it, round, g, tag, ctx->arrive);
    return;
  }
  if (!ctx->eval_v1) { /* second generation: one lane per pose */
    const bool wide = (long long)B * 2 <= 148; /* a CTA per band leaves SMs idle: give each band up to 16 warps */
    /* two compilations: <., 256> is built for 4 CTAs per SM (64 registers, a few spills) - what a full machine wants;
     * <., 512> keeps all 116 registers - faster per thread, right while every CTA is resident at 2 per SM anyway
     * (measured on C4: 128 / 256 bands 4.86 / 6.62 ms against 5.06 / 6.96; 512 bands 8.8 against 7.9 the other way) */
    const bool relaxed = wide || B <= 2 * 148;
    /* one warp per 30-pose tile of the longest band (2 .. 8 warps; 4 .. 16 in the wide variant: two trials side by side),
     * so that the K x tiles warp tasks split evenly and nobody idles at the barrier */
    int warps = ev2_tiles(db.n_cap);
    warps = warps < 2 ? 2 : (warps > 8 ? 8 : warps);
    if (wide) warps = 2 * warps;
    const int nt = 32 * warps;
    if (kp.generic) {
      if (relaxed) k_trial_eval2<true, 512><<<B, nt, smem, st>>>(db, kp, spec, it, round, g, tag);
      else k_trial_eval2<true, 256><<<B, nt, smem, st>>>(db, kp, spec, it, round, g, tag);
    } else {
      if (relaxed) k_trial_eval2<false, 512><<<B, nt, smem, st>>>(db, kp, spec, it, round, g, tag);
      else k_trial_eval2<false, 256><<<B, nt, smem, st>>>(db, kp, spec, it, round, g, tag);
    }
    return;
  }
  if (kp.generic) k_trial_eval<2, true><<<B, 32 * K, smem, st>>>(db, kp, spec, it, round, g, tag);
  else if (ctx->eval_minb == 3) k_trial_eval<3, false><<<B, 32 * K, smem, st>>>(db, kp, spec, it, round, g, tag);
  else k_trial_eval<2, false><<<B, 32 * K, smem, st>>>(db, kp, spec, it, round, g, tag);
}

/* The solve of one speculative round of solver 2: the B x K (band, trial) systems of round `round` of LM iteration `it`
 * (retry-list index g), with the mapping chosen by tebgpu_set_warp_solver - in the automatic modes by the number of
 * systems. Shared by issue_optimize and tebgpu_solve_system, so that the test entry point runs the optimizer's grid,
 * shared-memory size and kernel choice. Returns the number of kernels launched. */
static int launch_solve_kernel(const tebgpu_ctx* ctx, const DevBatch& db, const SpecBufs& spec, int B, int K, int it, int round,
                               int g, cudaStream_t s) {
  /* ring depth: 10 rows unless TEBGPU_RING asks for 20 / 30. Measured (profiles/r2_history.md): deeper rings do
   * not shorten the chain - a lone solver warp is bound by its own fp64 issue rate (~75 DFMA per pivot at 2
   * cycles each), not by the prefetch distance - and they cost residency (20 rows: 3 warps per SM). */
  const int bk = B * K;
  const int warps = (bk + 31) / 32;
  const int ring = ctx->ring == 0 ? 10 : ctx->ring;
  /* k_solve_warp: the sequential order spread over a warp (cross-check only) */
  const bool warp_solver = ctx->warp_solver == 1 || (ctx->warp_solver == 2 && bk <= 148 * 8);
  const size_t smem_lat = solve_lat_smem_bytes(db.n_cap);
  /* automatic: while the round's systems fit LAT_WAVES waves of resident CTAs (one warp + its whole system per CTA)
   * the twisted solver's ~0.065 ms per wave (200 poses) beats the 0.26 ms a thread-per-system solve takes
   * regardless of the count */
  const long long lat_wave = smem_lat <= 232448 ? 148LL * (232448 / smem_lat > 16 ? 16 : 232448 / smem_lat) : 0;
  const bool lat_solver = lat_wave > 0 && (ctx->warp_solver == 3 || (ctx->warp_solver == 4 && bk <= LAT_WAVES * lat_wave));
  if (lat_solver) k_solve_lat<<<bk, 32, smem_lat, s>>>(db, spec, it, round, g);
  else if (round > 0 && ctx->warp_solver == 4 && lat_wave > 0) {
    /* retry round of the throughput regime: both mappings are launched, the list length decides on the device */
    SpecBufs sl = spec;
    const long long cap = LAT_WAVES * lat_wave < bk ? LAT_WAVES * lat_wave : bk;
    sl.lat_cap = (int32_t)cap;
    k_solve_lat<<<(unsigned)cap, 32, smem_lat, s>>>(db, sl, it, round, g);
    k_solve_tpb<10><<<warps, 32, tpb_ring_bytes(10), s>>>(db, sl, it, round, g);
    return 2;
  }
  else if (warp_solver) k_solve_warp<<<(bk + SW_WARPS - 1) / SW_WARPS, 32 * SW_WARPS, 0, s>>>(db, spec, it, round, g);
  else if (ring == 30) k_solve_tpb<30><<<warps, 32, tpb_ring_bytes(30), s>>>(db, spec, it, round, g);
  else if (ring == 20) k_solve_tpb<20><<<warps, 32, tpb_ring_bytes(20), s>>>(db, spec, it, round, g);
  else k_solve_tpb<10><<<warps, 32, tpb_ring_bytes(10), s>>>(db, spec, it, round, g);
  return 1;
}

static KParams make_kparams(const tebgpu_ctx* ctx, const TebBatch* bt, double weight_multiplier) {
  const TebParams& p = ctx->params;
  KParams k;
  std::memset(&k, 0, sizeof(k));
  k.p = p;
  k.generic = p.footprint_type >= TEB_FOOTPRINT_LINE || bt->PV_cap > 0;
  k.fp_geom = ctx->d_fp;
  k.w_obst = p.weight_obstacle * weight_multiplier;
  k.sw_vel_x = std::sqrt(p.weight_max_vel_x); k.sw_vel_th = std::sqrt(p.weight_max_vel_theta);
  k.sw_acc_x = std::sqrt(p.weight_acc_lim_x); k.sw_acc_th = std::sqrt(p.weight_acc_lim_theta);
  k.inflated = p.inflation_dist > p.min_obstacle_dist;
  k.carlike = !(p.min_turning_radius == 0 || p.weight_kinematics_turning_radius == 0);
  k.sw_kin_nh = std::sqrt(p.weight_kinematics_nh);
  k.sw_kin_2 = std::sqrt(k.carlike ? p.weight_kinematics_turning_radius : p.weight_kinematics_forward_drive);
  k.sw_sp = std::sqrt(p.weight_shortest_path);
  k.sw_rot = std::sqrt(p.weight_prefer_rotdir);
  /* holonomic edge families: optimal_planner.cpp:722 / :745 (velocity), :778 / :824 (acceleration) */
  k.holo_vel = p.max_vel_y != 0;
  k.holo_acc = p.max_vel_y != 0 && p.acc_lim_y != 0;
  k.sw_vel_y = std::sqrt(p.weight_max_vel_y); k.sw_acc_y = std::sqrt(p.weight_acc_lim_y);
  k.has_vel = k.holo_vel ? !(p.weight_max_vel_x == 0 && p.weight_max_vel_y == 0 && p.weight_max_vel_theta == 0)
                         : !(p.weight_max_vel_x == 0 && p.weight_max_vel_theta == 0);
  k.has_acc = !(p.weight_acc_lim_x == 0 && p.weight_acc_lim_theta == 0); /* weight_acc_lim_y is not consulted (:768) */
  k.has_kin = k.carlike ? !(p.weight_kinematics_nh == 0 && p.weight_kinematics_turning_radius == 0)
                        : !(p.weight_kinematics_nh == 0 && p.weight_kinematics_forward_drive == 0);
  k.has_sp = p.weight_shortest_path != 0;
  k.has_rot = p.weight_prefer_rotdir != 0;
  k.has_time = p.weight_optimaltime != 0;
  k.has_obst = !(p.weight_obstacle == 0 || weight_multiplier == 0);
  k.has_dyn = p.include_dynamic_obstacles && p.weight_obstacle != 0; /* optimal_planner.cpp:342, :648 */
  k.has_via = p.weight_viapoint != 0;
  k.pow_exponent = (p.obstacle_cost_exponent != 1.0 && p.min_obstacle_dist > 0.0);
  /* optimal_planner.cpp:362; with the legacy association obstacles_per_vertex_ stays empty -> no ratio edges */
  k.has_vor = p.weight_velocity_obstacle_ratio > 0 && !p.legacy_obstacle_association;
  return k;
}

static int32_t check_batch(tebgpu_ctx* ctx, const TebBatch* bt) {
  if (!ctx || !bt) return TEBGPU_ERR_INVALID_ARG;
  if (bt->B < 1 || bt->n_cap < 3 || bt->S < 1 || bt->M_cap < 0 || bt->V_cap < 0) { ctx->err = "bad batch dimensions"; return TEBGPU_ERR_INVALID_ARG; }
  if (bt->B > ctx->lim.max_bands || bt->n_cap > ctx->lim.max_poses || bt->S > ctx->lim.max_scenes ||
      bt->M_cap > ctx->lim.max_obstacles || bt->V_cap > ctx->lim.max_viapoints) { ctx->err = "batch exceeds the context limits"; return TEBGPU_ERR_CAPACITY; }
  if (!bt->poses || !bt->n || !bt->scene_id || !bt->obst_count || !bt->vel_start || !bt->vel_goal) { ctx->err = "missing required batch array"; return TEBGPU_ERR_INVALID_ARG; }
  if (bt->M_cap > 0 && !bt->obstacles) { ctx->err = "obstacles == NULL"; return TEBGPU_ERR_INVALID_ARG; }
  if (bt->V_cap > 0 && (!bt->via || !bt->via_count)) { ctx->err = "via == NULL"; return TEBGPU_ERR_INVALID_ARG; }
  if (bt->PV_cap < 0 || bt->PV_cap > ctx->lim.max_obst_vertices) { ctx->err = "PV_cap exceeds max_obst_vertices"; return TEBGPU_ERR_CAPACITY; }
  if (bt->PV_cap > 0 && !bt->obst_vertices) { ctx->err = "obst_vertices == NULL"; return TEBGPU_ERR_INVALID_ARG; }
  if (!ctx->have_params) { ctx->err = "tebgpu_set_params has not been called"; return TEBGPU_ERR_INVALID_ARG; }
  return TEBGPU_OK;
}

static DevBatch make_devbatch(tebgpu_ctx* ctx, const TebBatch* bt) {
  DevBatch d;
  std::memset(&d, 0, sizeof(d));
  d.B = bt->B; d.n_cap = bt->n_cap; d.S = bt->S; d.M_cap = bt->M_cap; d.V_cap = bt->V_cap;
  d.MW = (bt->M_cap + 63) / 64; if (d.MW < 1) d.MW = 1;
  d.poses = bt->poses; d.n = bt->n; d.scene_id = bt->scene_id; d.obstacles = bt->obstacles; d.obst_count = bt->obst_count;
  d.via = bt->via; d.via_count = bt->via_count; d.vel_start = bt->vel_start; d.vel_goal = bt->vel_goal;
  d.prefer_rotdir = bt->prefer_rotdir;
  d.cost = bt->cost; d.chi2 = bt->chi2; d.status = bt->status; d.lm_iters = bt->lm_iters;
  d.Hb = ctx->Hb; d.assoc = ctx->assoc; d.assoc3 = ctx->assoc3; d.dyn_t = ctx->dyn_t; d.via_idx = ctx->via_idx; d.chi_parts = ctx->chi_parts; d.dmax_parts = ctx->dmax_parts; d.rhs = ctx->rhs; d.dyn_idx = ctx->dyn_idx; d.dyn_cnt = ctx->dyn_cnt;
  d.state = ctx->state;
  d.tile = ctx->linearize_variant == 1 ? TP : KA2_TP;
  d.chunks = (bt->n_cap + d.tile - 1) / d.tile;
  d.obst_vertices = bt->PV_cap > 0 ? bt->obst_vertices : nullptr; d.PV_cap = bt->PV_cap;
  d.defer = ctx->defer; d.a_list = nullptr; d.a_cnt = nullptr; d.skip_tag = 0;
  return d;
}

/* the launch sequence of one optimizeTEB over the batch, issued on `st` (directly, or into a stream capture) */
static int32_t issue_optimize(tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* args, cudaStream_t st) {
  DevBatch db = make_devbatch(ctx, bt);
  const TebParams& p = ctx->params;
  const int B = bt->B;
  const int tb = 128, gb = ((B > bt->S ? B : bt->S) + tb - 1) / tb;
  int64_t launches = 0;
  const size_t smem_a = ka_smem_bytes(bt->M_cap);
  const size_t smem_b = kb_smem_bytes(bt->n_cap, bt->M_cap);
  const size_t smem_bcr = kb_bcr_smem_bytes(bt->n_cap, bt->M_cap);
  const bool use_bcr = ctx->solver == 1 && bt->n_cap <= BCR_MAX_POSES && smem_bcr <= 232448 &&
                       ctx->lim.max_poses <= BCR_MAX_POSES;
  const size_t smem_g = (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) * sizeof(TebObstacle);
  /* speculation width: one solver warp per SM sub-partition is the latency-optimal regime (148 SMs x 4 x 32 lanes);
   * below it the wider speculation is free and removes the second round, above it the factor traffic dominates */
  /* Speculation schedule: widths of the rounds of one LM iteration (they add up to g2o's 10 trials).
   *   fixed width (tebgpu_set_speculation / TEBGPU_SPEC_K): K, K, ... as before;
   *   automatic: the first LM iteration after every graph rebuild restarts at lambda = 1e-5 max diag and needs 4-5
   *   damping escalations on 90 % of the bands, later iterations accept the first trial on 60 % (measured on C2-C4,
   *   profiles/r2_history.md). Latency regime (all B x 8 systems fit one solver warp per SM sub-partition): {8, 2} -
   *   the retry round practically never runs. Throughput regime: {6, 4} for the first iteration, {2, 4, 4} afterwards
   *   - factor traffic and trial evaluations follow the width. */
  int sched_first[5] = {0, 0, 0, 0, 0}, sched_later[5] = {0, 0, 0, 0, 0};
  int n_first = 0, n_later = 0;
  {
    int kmax = SPEC_K_MAX;
    while (kmax > 2 && eval_bytes(ctx, bt->n_cap, bt->M_cap, kmax) > 232448) kmax -= 2;
    if (eval_bytes(ctx, bt->n_cap, bt->M_cap, kmax) > 232448) { ctx->err = "trial-evaluation staging exceeds shared memory"; return TEBGPU_ERR_CAPACITY; }
    auto fill = [&](int* dst, int& cnt, std::initializer_list<int> want) {
      int left = 10;
      cnt = 0;
      for (int w : want) {
        if (left <= 0) break;
        int k = w < kmax ? w : kmax;
        dst[cnt++] = k;
        left -= k;
      }
      while (left > 0) { dst[cnt++] = kmax < 4 ? kmax : 4; left -= dst[cnt - 1]; }
    };
    if (ctx->spec_k != 0) {
      const int k = ctx->spec_k;
      fill(sched_first, n_first, {k, k, k, k, k});
      fill(sched_later, n_later, {k, k, k, k, k});
    } else if ((long long)B * 8 <= 148LL * 4 * 32) {
      fill(sched_first, n_first, {8, 2});
      fill(sched_later, n_later, {8, 2});
    } else {
      fill(sched_first, n_first, {6, 4});
      fill(sched_later, n_later, {2, 4, 4});
    }
  }
  const int rounds_max = n_first > n_later ? n_first : n_later;
  ctx->last_spec_k = ctx->solver == 2 ? sched_later[0] : 1;
  ctx->last_spec_first = ctx->solver == 2 ? sched_first[0] : 1;
  int g = 0; /* running index of the speculative rounds of this call: selects the retry-list counter / buffer */
  if (ctx->solver == 2) {
    const long long need_cnt = (long long)args->iterations_outerloop * args->iterations_innerloop * rounds_max + 2;
    if (need_cnt > SPEC_CNT_CAP) { ctx->err = "outer x inner iterations exceed the retry-list counters"; return TEBGPU_ERR_CAPACITY; }
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->spec.cnt, 0, (size_t)need_cnt * sizeof(int32_t), st));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->defer, 0, (size_t)B * sizeof(int32_t), st));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->arrive, 0, (size_t)B * sizeof(int32_t), st)); /* k_trial_eval3's arrival counters: a call that
                                                                                    was cut short must not leak into the next */
  }
  /* Retry rounds (bands that rejected all trials of a round) can run on a side stream, followed by kernel A of the next
   * inner iteration for exactly those bands - and, with TEBGPU_SPLIT, by ROUND 0 of that iteration for them - while the
   * main stream works on all other bands. Bands never share data, so this is only a re-ordering of independent work
   * (bit-identical results, tested). It pays when the retry rounds are nearly empty (fixed K = 4: ~5 % of the bands; the
   * latency regime, where it is the default). With the width schedule {2, 4, 4} of the throughput regime 30-40 % of the
   * bands retry, the retry solves move as many factor bytes as round 0, and the overlapped schedules measure within
   * +-3 % of the serial one on C2 / C3 / C4 (profiles/r2_history.md): the machine is resource bound, so one stream is the
   * default there. */
  const bool latency_regime_b = (long long)B * 8 <= 148LL * 4 * 32;
  const bool overlap = ctx->solver == 2 && (ctx->overlap == 1 || (ctx->overlap == 2 && latency_regime_b)) && !ctx->profiling;
  int tag = 0; /* running inner-iteration number (1-based) */
  double weight_multiplier = 1.0;
  KParams kp = make_kparams(ctx, bt, weight_multiplier);
  prof_begin(ctx, st, 0); k_begin<<<gb, tb, 0, st>>>(db, kp); ++launches; prof_end(ctx, st);
  const bool split_ok = overlap && ctx->split && !latency_regime_b;
  bool side_share = false;
  int last_r1 = 0;      /* index g of round 1 of the latest LM iteration: its list = the side stream's bands */
  bool carried = false; /* the side stream already ran autoResize / buildGraph / kernel A of this outer iteration for the
                           bands that were still in a retry round when the previous outer iteration ended */
  for (int o = 0; o < args->iterations_outerloop; ++o) {
    kp = make_kparams(ctx, bt, weight_multiplier);
    {
      DevBatch dm = db;
      if (carried) dm.skip_tag = tag;
      if (p.teb_autosize) { prof_begin(ctx, st, 1); k_auto_resize<<<gb, tb, 0, st>>>(dm, kp); ++launches; prof_end(ctx, st); }
      prof_begin(ctx, st, 2); launch_build_graph(dm, kp, B, smem_g, st); ++launches; prof_end(ctx, st);
    }
    bool deferred_done = carried; /* kernel A of this iteration already ran for the deferred bands (side stream) */
    carried = false;
    for (int it = 0; it < args->iterations_innerloop; ++it) {
      ++tag;
      {
        DevBatch da = db;
        if (deferred_done) da.skip_tag = tag - 1; /* bands queued during the previous iteration were linearised on the side stream */
        prof_begin(ctx, st, 3); launch_linearize(ctx, da, kp, B, bt->M_cap, st); ++launches; prof_end(ctx, st);
        if (kp.has_vor) { prof_begin(ctx, st, 3); launch_vor(db, kp, B, smem_g, st); ++launches; prof_end(ctx, st); }
        /* Split round 0 (throughput regime): the bands that needed retry rounds in the previous iteration were linearised
         * on the side stream; instead of joining here, the side stream also solves / evaluates ROUND 0 for exactly those
         * bands (list of the previous round 1, own scratch) while the main stream does it for all others. Both append to
         * the same retry list; the main stream waits for the side stream's evaluation only before it needs the deferral
         * tags again. Bands never share data: only the schedule changes, the results do not. */
        side_share = deferred_done && split_ok;
        if (deferred_done && !side_share) CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
        deferred_done = false;
      }
      if (ctx->solver == 2) {
        const int* sched = (it == 0) ? sched_first : sched_later;
        const int rounds = (it == 0) ? n_first : n_later; /* widths add up to g2o's maxTrialsAfterFailure = 10 */
        const bool fork = overlap && rounds > 1 && !kp.has_vor;
        cudaStream_t rs = st;
        auto launch_solve = [&](const SpecBufs& spec, int K, int round, cudaStream_t s) {
          launches += launch_solve_kernel(ctx, db, spec, B, K, it, round, g, s);
        };
        for (int round = 0; round < rounds; ++round, ++g) {
          const int K = sched[round];
          ctx->spec.K = K;
          const size_t smem_e = eval_bytes(ctx, bt->n_cap, bt->M_cap, K);
          SpecBufs spec = ctx->spec; /* main-stream launch: every band, or every band but the side stream's share */
          if (round == 0 && side_share) { spec.defer = ctx->defer; spec.skip_tag = tag - 1; }
          if (round == 1 && fork) { /* retry rounds go to the side stream */
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, st));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0));
            rs = ctx->side;
          }
          if (rs == ctx->side) { spec.Lf = ctx->Lf2; spec.dx = ctx->dx2; } /* the side stream's own scratch */
          if (round == 0 && side_share) { /* the side stream's share of round 0, issued before its retry rounds */
            SpecBufs ss = ctx->spec;
            ss.Lf = ctx->Lf2; ss.dx = ctx->dx2;
            ss.sel_list = ctx->spec.list + (size_t)(last_r1 % SPEC_LISTS) * B;
            ss.sel_cnt = ctx->spec.cnt + last_r1;
            launch_solve(ss, K, 0, ctx->side);
            launch_trial_eval(ctx, ss, db, kp, B, K, smem_e, it, 0, g, tag, ctx->side); ++launches;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_s0, ctx->side));
          }
          prof_begin(ctx, st, round == 0 ? 6 : 4);
          launch_solve(spec, K, round, rs);
          prof_end(ctx, st);
          prof_begin(ctx, st, round == 0 ? 7 : 4);
          launch_trial_eval(ctx, spec, db, kp, B, K, smem_e, it, round, g, tag, rs);
          ++launches; prof_end(ctx, st);
          /* the deferral tags / the retry list of this iteration are complete once both halves of round 0 are done */
          if (round == 0 && side_share) CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_s0, 0));
        }
        last_r1 = g - rounds + 1;
        if (fork) {
          if (it + 1 < args->iterations_innerloop) { /* next kernel A for the bands of the round-1 list, then join */
            DevBatch dl = db;
            dl.a_list = ctx->spec.list + (size_t)(last_r1 % SPEC_LISTS) * B;
            dl.a_cnt = ctx->spec.cnt + last_r1;
            launch_linearize(ctx, dl, kp, B, bt->M_cap, ctx->side); ++launches;
            deferred_done = true;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->side));
          } else if (o + 1 < args->iterations_outerloop) {
            /* last inner iteration: the side stream goes on with the next outer iteration's autoResize / buildGraph /
             * first kernel A for its bands (next weight multiplier), the main stream does the same for all others */
            const KParams kn = make_kparams(ctx, bt, weight_multiplier * p.weight_adapt_factor);
            DevBatch dl = db;
            dl.a_list = ctx->spec.list + (size_t)(last_r1 % SPEC_LISTS) * B;
            dl.a_cnt = ctx->spec.cnt + last_r1;
            if (p.teb_autosize) { k_auto_resize<<<gb, tb, 0, ctx->side>>>(dl, kn); ++launches; }
            launch_build_graph(dl, kn, B, smem_g, ctx->side); ++launches;
            launch_linearize(ctx, dl, kn, B, bt->M_cap, ctx->side); ++launches;
            carried = true;
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->side));
          } else {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->side));
            CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
          }
        }
      } else {
        prof_begin(ctx, st, 4);
        if (use_bcr && kp.generic) k_lm_step_t<1, KB_BCR_THREADS, true><<<B, KB_BCR_THREADS, smem_bcr, st>>>(db, kp, it);
        else if (use_bcr) k_lm_step_t<1, KB_BCR_THREADS, false><<<B, KB_BCR_THREADS, smem_bcr, st>>>(db, kp, it);
        else if (kp.generic) k_lm_step_t<0, KB_THREADS, true><<<B, KB_THREADS, smem_b, st>>>(db, kp, it);
        else k_lm_step_t<0, KB_THREADS, false><<<B, KB_THREADS, smem_b, st>>>(db, kp, it);
        ++launches; prof_end(ctx, st);
      }
    }
    weight_multiplier *= p.weight_adapt_factor; /* optimal_planner.cpp:227 */
  }
  prof_begin(ctx, st, 5); k_finalize<<<gb, tb, 0, st>>>(db, kp, *args); ++launches; prof_end(ctx, st);
  ctx->launches = launches;
  if (ctx->profiling && ctx->ev_used > 4096) { cudaStreamSynchronize(st); prof_collect(ctx); }
  CUDA_TRY(ctx, cudaGetLastError());
  return TEBGPU_OK;
}

/* CUDA-graph replay of the launch sequence. The sequence is a pure function of the batch description (dimensions and
 * buffer addresses), the optimize arguments, the parameter block and the context switches, so it is captured once per
 * distinct key (fork / join of the retry side stream included) and replayed afterwards: one graph launch instead of
 * ~130-170 kernel launches. That only matters in the latency regime (a single planning request: kernels of 10-50 us), so
 * graphs are used there by default (tebgpu_set_graph: 0 never, 1 always, 2 automatic). */
static uint64_t graph_key(const tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* a, cudaStream_t st) {
  uint64_t h = 1469598103934665603ull;
  auto mix = [&](const void* p, size_t nbytes) {
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t k = 0; k < nbytes; ++k) { h ^= c[k]; h *= 1099511628211ull; }
  };
  mix(bt, sizeof(*bt));
  mix(a, sizeof(*a));
  mix(&ctx->params_version, sizeof(ctx->params_version));
  const int sw[11] = {ctx->solver, ctx->spec_k, ctx->linearize_variant, ctx->ka_staged, ctx->eval_v1, ctx->ring, ctx->overlap, ctx->eval_minb, ctx->warp_solver, ctx->eval_mode, ctx->split};
  mix(sw, sizeof(sw));
  mix(&st, sizeof(st));
  return h;
}

int32_t tebgpu_optimize_batch_device(tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* args, void* cuda_stream) {
  int32_t rc = check_batch(ctx, bt);
  if (rc) return rc;
  if (!args || args->iterations_innerloop < 0 || args->iterations_outerloop < 0) { ctx->err = "bad optimize args"; return TEBGPU_ERR_INVALID_ARG; }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : ctx->stream;
  const bool latency_regime = (long long)bt->B * 8 <= 148LL * 4 * 32;
  const bool use_graph = !ctx->profiling && (ctx->graph_mode == 1 || (ctx->graph_mode == 2 && latency_regime));
  if (!use_graph) return issue_optimize(ctx, bt, args, st);
  const uint64_t key = graph_key(ctx, bt, args, st);
  for (auto& e : ctx->graphs)
    if (e.key == key) {
      e.stamp = ++ctx->graph_clock;
      ctx->launches = e.launches;
      ctx->last_spec_k = e.spec_k; ctx->last_spec_first = e.spec_first;
      CUDA_TRY(ctx, cudaGraphLaunch(e.exec, st));
      return TEBGPU_OK;
    }
  CUDA_TRY(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  rc = issue_optimize(ctx, bt, args, st);
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(st, &graph);
  if (rc != TEBGPU_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    if (rc == TEBGPU_OK) { /* capture itself failed: run the sequence directly */
      ctx->graph_mode = 0;
      return issue_optimize(ctx, bt, args, st);
    }
    return rc;
  }
  tebgpu_ctx::GraphEntry ent;
  ent.key = key; ent.launches = ctx->launches; ent.stamp = ++ctx->graph_clock;
  ent.spec_k = ctx->last_spec_k; ent.spec_first = ctx->last_spec_first;
  const cudaError_t ie = cudaGraphInstantiate(&ent.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) { cudaGetLastError(); ctx->graph_mode = 0; return issue_optimize(ctx, bt, args, st); }
  if (ctx->graphs.size() >= 8) { /* drop the least recently used graph */
    size_t old = 0;
    for (size_t k = 1; k < ctx->graphs.size(); ++k)
      if (ctx->graphs[k].stamp < ctx->graphs[old].stamp) old = k;
    cudaGraphExecDestroy(ctx->graphs[old].exec);
    ctx->graphs.erase(ctx->graphs.begin() + old);
  }
  ctx->graphs.push_back(ent);
  CUDA_TRY(ctx, cudaGraphLaunch(ent.exec, st));
  return TEBGPU_OK;
}

int32_t tebgpu_set_warp_solver(tebgpu_ctx* ctx, int32_t mode) {
  if (!ctx || mode < 0 || mode > 4) return TEBGPU_ERR_INVALID_ARG;
  ctx->warp_solver = mode;
  return TEBGPU_OK;
}

int32_t tebgpu_set_graph(tebgpu_ctx* ctx, int32_t mode) {
  if (!ctx || mode < 0 || mode > 2) return TEBGPU_ERR_INVALID_ARG;
  ctx->graph_mode = mode;
  return TEBGPU_OK;
}

int32_t tebgpu_set_profiling(tebgpu_ctx* ctx, int32_t enable) {
  if (!ctx) return TEBGPU_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  prof_collect(ctx);
  ctx->profiling = enable != 0;
  for (int k = 0; k < 9; ++k) { ctx->prof_ms[k] = 0; ctx->prof_cnt[k] = 0; }
  return TEBGPU_OK;
}

int32_t tebgpu_get_kernel_times(tebgpu_ctx* ctx, double ms_out[9], int64_t count_out[9]) {
  if (!ctx || !ms_out || !count_out) return TEBGPU_ERR_INVALID_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  prof_collect(ctx);
  for (int k = 0; k < 9; ++k) { ms_out[k] = ctx->prof_ms[k]; count_out[k] = ctx->prof_cnt[k]; ctx->prof_ms[k] = 0; ctx->prof_cnt[k] = 0; }
  return TEBGPU_OK;
}

int32_t tebgpu_set_linearize_variant(tebgpu_ctx* ctx, int32_t v) {
  if (!ctx || v < 0 || v > 1) return TEBGPU_ERR_INVALID_ARG;
  ctx->linearize_variant = v;
  return TEBGPU_OK;
}

int32_t tebgpu_set_speculation(tebgpu_ctx* ctx, int32_t k) {
  if (!ctx || !(k == 0 || k == 2 || k == 4 || k == 6 || k == 8)) return TEBGPU_ERR_INVALID_ARG;
  ctx->spec_k = k;
  return TEBGPU_OK;
}

int32_t tebgpu_set_solver(tebgpu_ctx* ctx, int32_t solver) {
  if (!ctx || solver < 0 || solver > 2) return TEBGPU_ERR_INVALID_ARG;
  ctx->solver = solver;
  return TEBGPU_OK;
}

int32_t tebgpu_synchronize(tebgpu_ctx* ctx) {
  if (!ctx) return TEBGPU_ERR_INVALID_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return TEBGPU_OK;
}

static TebBatch mirror_batch(tebgpu_ctx* ctx, const TebBatch* bt) {
  TebBatch d = *bt;
  d.poses = ctx->d_poses; d.n = ctx->d_n; d.scene_id = ctx->d_scene; d.obstacles = ctx->d_obst; d.obst_count = ctx->d_ocount;
  d.via = bt->V_cap > 0 ? ctx->d_via : nullptr; d.via_count = bt->V_cap > 0 ? ctx->d_vcount : nullptr;
  d.vel_start = ctx->d_vs; d.vel_goal = ctx->d_vg; d.prefer_rotdir = bt->prefer_rotdir ? ctx->d_rot : nullptr;
  d.cost = ctx->d_cost; d.chi2 = ctx->d_chi2; d.status = ctx->d_status; d.lm_iters = ctx->d_iters;
  d.obst_vertices = bt->PV_cap > 0 ? ctx->d_pverts : nullptr;
  return d;
}

static int32_t upload_batch(tebgpu_ctx* ctx, const TebBatch* bt) {
  cudaStream_t st = ctx->stream;
  const size_t B = bt->B, nc = bt->n_cap;
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_poses, bt->poses, B * nc * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_n, bt->n, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_scene, bt->scene_id, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (bt->M_cap > 0)
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_obst, bt->obstacles, (size_t)bt->S * bt->M_cap * sizeof(TebObstacle), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_ocount, bt->obst_count, (size_t)bt->S * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (bt->PV_cap > 0)
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_pverts, bt->obst_vertices, (size_t)bt->S * bt->PV_cap * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
  /* host entry points can check every per-element input before the device indexes with it */
  for (int sc = 0; sc < bt->S; ++sc)
    if (bt->obst_count[sc] < 0 || bt->obst_count[sc] > bt->M_cap) { ctx->err = "obst_count[s] outside 0 .. M_cap"; return TEBGPU_ERR_INVALID_ARG; }
  for (int b = 0; b < bt->B; ++b) {
    if (bt->scene_id[b] < 0 || bt->scene_id[b] >= bt->S) { ctx->err = "scene_id[b] outside 0 .. S-1"; return TEBGPU_ERR_INVALID_ARG; }
    if (bt->n[b] < 0 || bt->n[b] > bt->n_cap) { ctx->err = "n[b] outside 0 .. n_cap"; return TEBGPU_ERR_INVALID_ARG; }
    if (bt->V_cap > 0 && (bt->via_count[b] < 0 || bt->via_count[b] > bt->V_cap)) { ctx->err = "via_count[b] outside 0 .. V_cap"; return TEBGPU_ERR_INVALID_ARG; }
  }
  for (int sc = 0; sc < bt->S; ++sc)
    for (int m = 0; m < bt->obst_count[sc] && m < bt->M_cap; ++m) {
      const TebObstacle& o = bt->obstacles[(size_t)sc * bt->M_cap + m];
      if (o.type < TEB_OBST_POINT || o.type > TEB_OBST_POLYGON) { ctx->err = "unknown obstacle type"; return TEBGPU_ERR_INVALID_ARG; }
      if (o.type >= TEB_OBST_LINE) {
        const int need = o.type == TEB_OBST_POLYGON ? 1 : 2;
        if (o.vertex_count < need || (o.type != TEB_OBST_POLYGON && o.vertex_count != 2) || o.vertex_begin < 0 ||
            (long long)o.vertex_begin + o.vertex_count > bt->PV_cap) {
          ctx->err = "obstacle vertex range outside obst_vertices";
          return TEBGPU_ERR_INVALID_ARG;
        }
      }
    }
  if (bt->V_cap > 0) {
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_via, bt->via, B * bt->V_cap * 2 * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vcount, bt->via_count, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vs, bt->vel_start, B * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_vg, bt->vel_goal, B * 4 * sizeof(double), cudaMemcpyHostToDevice, st));
  if (bt->prefer_rotdir)
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_rot, bt->prefer_rotdir, B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  return TEBGPU_OK;
}

int32_t tebgpu_optimize_batch(tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* args) {
  int32_t rc = check_batch(ctx, bt);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  rc = upload_batch(ctx, bt);
  if (rc) return rc;
  TebBatch d = mirror_batch(ctx, bt);
  rc = tebgpu_optimize_batch_device(ctx, &d, args, nullptr);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const size_t B = bt->B, nc = bt->n_cap;
  CUDA_TRY(ctx, cudaMemcpyAsync(bt->poses, ctx->d_poses, B * nc * 4 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(bt->n, ctx->d_n, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (bt->cost) CUDA_TRY(ctx, cudaMemcpyAsync(bt->cost, ctx->d_cost, B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (bt->chi2) CUDA_TRY(ctx, cudaMemcpyAsync(bt->chi2, ctx->d_chi2, B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (bt->status) CUDA_TRY(ctx, cudaMemcpyAsync(bt->status, ctx->d_status, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (bt->lm_iters) CUDA_TRY(ctx, cudaMemcpyAsync(bt->lm_iters, ctx->d_iters, B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return TEBGPU_OK;
}

int32_t tebgpu_compute_cost(tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* args) {
  int32_t rc = check_batch(ctx, bt);
  if (rc) return rc;
  if (!args) return TEBGPU_ERR_INVALID_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  rc = upload_batch(ctx, bt);
  if (rc) return rc;
  TebBatch d = mirror_batch(ctx, bt);
  cudaStream_t st = ctx->stream;
  DevBatch db = make_devbatch(ctx, &d);
  KParams kp = make_kparams(ctx, bt, 1.0); /* buildGraph() default weight_multiplier (optimal_planner.h:536) */
  const int B = bt->B, tb = 128, gb = ((B > bt->S ? B : bt->S) + tb - 1) / tb;
  k_begin<<<gb, tb, 0, st>>>(db, kp);
  launch_build_graph(db, kp, B, (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) * sizeof(TebObstacle), st);
  launch_linearize(ctx, db, kp, B, bt->M_cap, st);
  if (kp.has_vor) launch_vor(db, kp, B, (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) * sizeof(TebObstacle), st);
  k_cost_only<<<gb, tb, 0, st>>>(db, kp, *args);
  ctx->launches = 4;
  CUDA_TRY(ctx, cudaGetLastError());
  if (bt->cost) CUDA_TRY(ctx, cudaMemcpyAsync(bt->cost, ctx->d_cost, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (bt->chi2) CUDA_TRY(ctx, cudaMemcpyAsync(bt->chi2, ctx->d_chi2, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (bt->status) CUDA_TRY(ctx, cudaMemcpyAsync(bt->status, ctx->d_status, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return TEBGPU_OK;
}

int32_t tebgpu_h_signature(tebgpu_ctx* ctx, const TebBatch* bt, int32_t use_timediffs, double* h_out, int32_t device_ptrs) {
  int32_t rc = check_batch(ctx, bt);
  if (rc) return rc;
  if (!h_out) return TEBGPU_ERR_INVALID_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  TebBatch d = *bt;
  if (!device_ptrs) {
    rc = upload_batch(ctx, bt);
    if (rc) return rc;
    d = mirror_batch(ctx, bt);
  }
  cudaStream_t st = ctx->stream;
  DevBatch db = make_devbatch(ctx, &d);
  KParams kp = make_kparams(ctx, bt, 1.0);
  const int B = bt->B;
  const bool three_d = ctx->params.include_dynamic_obstacles != 0; /* homotopy_class_planner.hpp:50 */
  const size_t stride = three_d ? (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) : 2;
  const size_t smem = hsig_smem_bytes(bt->n_cap, bt->M_cap);
  if (smem > 232448) { ctx->err = "h-signature staging exceeds shared memory"; return TEBGPU_ERR_CAPACITY; }
  double* d_out = device_ptrs ? h_out : ctx->d_hsig; /* [B][stride] <= [max_bands][max(max_obstacles, 2)] */
  if (three_d) {
    CUDA_TRY(ctx, cudaFuncSetAttribute(k_hsig3d, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_hsig3d<<<B, HSIG_THREADS, smem, st>>>(db, kp, use_timediffs, d_out);
  } else {
    CUDA_TRY(ctx, cudaFuncSetAttribute(k_hsig2d, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_hsig2d<<<B, HSIG_THREADS, smem, st>>>(db, kp, d_out);
  }
  ctx->launches = 1;
  CUDA_TRY(ctx, cudaGetLastError());
  if (!device_ptrs) {
    CUDA_TRY(ctx, cudaMemcpyAsync(h_out, d_out, (size_t)B * stride * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
  }
  return TEBGPU_OK;
}

int32_t tebgpu_build_system(tebgpu_ctx* ctx, const TebBatch* bt, int32_t outer_index, double* Hb_out, double* chi2_out,
                            int32_t device_ptrs) {
  int32_t rc = check_batch(ctx, bt);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  TebBatch d = *bt;
  if (!device_ptrs) {
    rc = upload_batch(ctx, bt);
    if (rc) return rc;
    d = mirror_batch(ctx, bt);
  }
  cudaStream_t st = ctx->stream;
  DevBatch db = make_devbatch(ctx, &d);
  double mult = 1.0;
  for (int o = 0; o < outer_index; ++o) mult *= ctx->params.weight_adapt_factor;
  KParams kp = make_kparams(ctx, bt, mult);
  const int B = bt->B, tb = 128, gb = ((B > bt->S ? B : bt->S) + tb - 1) / tb;
  k_begin<<<gb, tb, 0, st>>>(db, kp);
  launch_build_graph(db, kp, B, (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) * sizeof(TebObstacle), st);
  launch_linearize(ctx, db, kp, B, bt->M_cap, st);
  if (kp.has_vor) launch_vor(db, kp, B, (size_t)(bt->M_cap > 0 ? bt->M_cap : 1) * sizeof(TebObstacle), st);
  ctx->launches = 3;
  CUDA_TRY(ctx, cudaGetLastError());
  const size_t per_band = (size_t)4 * bt->n_cap * HROW;
  if (Hb_out)
    CUDA_TRY(ctx, cudaMemcpyAsync(Hb_out, ctx->Hb, (size_t)B * per_band * sizeof(double),
                                  device_ptrs ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  if (chi2_out) {
    /* sum the tile partials on the host side of the call */
    std::string hold;
    const size_t cnt = (size_t)B * db.chunks * 4;
    double* tmp = new (std::nothrow) double[cnt];
    int32_t* hn = new (std::nothrow) int32_t[B];
    if (!tmp || !hn) { delete[] tmp; delete[] hn; return TEBGPU_ERR_CUDA; }
    cudaError_t e1 = cudaMemcpyAsync(tmp, ctx->chi_parts, cnt * sizeof(double), cudaMemcpyDeviceToHost, st);
    cudaError_t e2 = cudaMemcpyAsync(hn, d.n, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    cudaError_t e3 = cudaStreamSynchronize(st);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) { delete[] tmp; delete[] hn; ctx->err = "chi2 readback failed"; return TEBGPU_ERR_CUDA; }
    double* host_chi = device_ptrs ? new (std::nothrow) double[B] : chi2_out;
    for (int b = 0; b < B; ++b) {
      double s = 0;
      const int used = (hn[b] + db.tile - 1) / db.tile;
      for (int c = 0; c < used; ++c)
        for (int k = 0; k < 4; ++k) s += tmp[((size_t)b * db.chunks + c) * 4 + k];
      host_chi[b] = s;
    }
    if (device_ptrs) {
      cudaMemcpy(chi2_out, host_chi, (size_t)B * sizeof(double), cudaMemcpyHostToDevice);
      delete[] host_chi;
    }
    delete[] tmp;
    delete[] hn;
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return TEBGPU_OK;
}

int32_t tebgpu_solve_system(tebgpu_ctx* ctx, int32_t B, int32_t n_cap, const int32_t* n, const double* Hb, const double* lambda,
                            const double* ni, int32_t K, double* dx_out, int32_t* ok_out, double* lambda_out) {
  if (!ctx || !n || !Hb || !lambda || !ni || !dx_out || !ok_out || !lambda_out) return TEBGPU_ERR_INVALID_ARG;
  if (B < 1 || n_cap < 3 || K < 1 || K > SPEC_K_MAX) { ctx->err = "bad solve dimensions"; return TEBGPU_ERR_INVALID_ARG; }
  if (B > ctx->lim.max_bands || n_cap > ctx->lim.max_poses) { ctx->err = "solve exceeds the context limits"; return TEBGPU_ERR_CAPACITY; }
  for (int b = 0; b < B; ++b)
    if (n[b] < 3 || n[b] > n_cap) { ctx->err = "n[b] outside 3 .. n_cap"; return TEBGPU_ERR_INVALID_ARG; }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t rows = (size_t)4 * n_cap;
  std::vector<BandState> hs((size_t)B);
  for (int b = 0; b < B; ++b) {
    std::memset(&hs[b], 0, sizeof(BandState));
    hs[b].active = 1;
    hs[b].lambda = lambda[b];
    hs[b].ni = ni[b];
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->Hb, Hb, (size_t)B * rows * HROW * sizeof(double), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_n, n, (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->state, hs.data(), (size_t)B * sizeof(BandState), cudaMemcpyHostToDevice, st));
  DevBatch db;
  std::memset(&db, 0, sizeof(db));
  db.B = B; db.n_cap = n_cap; db.n = ctx->d_n; db.Hb = ctx->Hb; db.state = ctx->state;
  db.tile = KA2_TP; db.chunks = (n_cap + KA2_TP - 1) / KA2_TP; db.dmax_parts = ctx->dmax_parts; db.defer = ctx->defer;
  SpecBufs spec = ctx->spec; /* round 0, no selection list: system t = K b + k */
  spec.K = K; spec.sel_list = nullptr; spec.sel_cnt = nullptr; spec.defer = nullptr; spec.skip_tag = 0; spec.lat_cap = 0;
  /* the solution scratch is filled with NaN first: rows a kernel does not write (4 n[b] .. 4 n_cap - 1, and the whole
   * system after a failed factorisation in the modes that stop there) come back as NaN */
  const int warps = (B * K + 31) / 32;
  const size_t dx_elems = (size_t)warps * 32 * rows;
  CUDA_TRY(ctx, cudaMemsetAsync(spec.dx, 0xff, dx_elems * sizeof(double), st));
  CUDA_TRY(ctx, cudaMemsetAsync(spec.res, 0, (size_t)B * SPEC_K_MAX * RES_STRIDE * sizeof(double), st));
  ctx->launches = launch_solve_kernel(ctx, db, spec, B, K, /*it=*/1, /*round=*/0, /*g=*/0, st);
  CUDA_TRY(ctx, cudaGetLastError());
  std::vector<double> hdx(dx_elems), hres((size_t)B * SPEC_K_MAX * RES_STRIDE);
  CUDA_TRY(ctx, cudaMemcpyAsync(hdx.data(), spec.dx, dx_elems * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(hres.data(), spec.res, hres.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  /* de-interleave: system t = K b + k sits in lane t & 31 of solver warp t >> 5, row r at [r][lane] */
  for (int b = 0; b < B; ++b)
    for (int k = 0; k < K; ++k) {
      const size_t t = (size_t)K * b + k;
      const double* src = hdx.data() + (t >> 5) * 32 * rows + (t & 31);
      double* dst = dx_out + t * rows;
      for (size_t r = 0; r < rows; ++r) dst[r] = src[r * 32];
      const double* res = hres.data() + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;
      ok_out[t] = res[5] != 0.0 ? 1 : 0;
      lambda_out[t] = res[6];
    }
  return TEBGPU_OK;
}

/* ------------------------------------------------------------------ the one collective: all-gather of the costs */
#define NCCL_TRY(ctx, expr)                                                                              \
  do {                                                                                                   \
    ncclResult_t _r = (expr);                                                                            \
    if (_r != ncclSuccess) {                                                                             \
      (ctx)->err = std::string(#expr) + ": " + (nccl_api().GetErrorString ? nccl_api().GetErrorString(_r) : "NCCL error"); \
      return TEBGPU_ERR_CUDA;                                                                            \
    }                                                                                                    \
  } while (0)

int32_t tebgpu_comm_get_unique_id(void* id_out) {
  static_assert(sizeof(ncclUniqueId) == TEBGPU_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
  if (!id_out) return TEBGPU_ERR_INVALID_ARG;
  NcclApi& api = nccl_api();
  if (!api.ok()) { std::fprintf(stderr, "tebgpu_comm_get_unique_id: %s\n", api.error.c_str()); return TEBGPU_ERR_UNSUPPORTED; }
  ncclUniqueId id;
  if (api.GetUniqueId(&id) != ncclSuccess) return TEBGPU_ERR_CUDA;
  std::memcpy(id_out, &id, sizeof(id));
  return TEBGPU_OK;
}

int32_t tebgpu_comm_init(tebgpu_ctx* ctx, const void* id, int32_t world_size, int32_t rank) {
  if (!ctx || !id || world_size < 1 || rank < 0 || rank >= world_size) return TEBGPU_ERR_INVALID_ARG;
  NcclApi& api = nccl_api();
  if (!api.ok()) { ctx->err = api.error.empty() ? "NCCL unavailable" : api.error; return TEBGPU_ERR_UNSUPPORTED; }
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  if (ctx->comm) { api.CommDestroy(ctx->comm); ctx->comm = nullptr; }
  ncclUniqueId uid;
  std::memcpy(&uid, id, sizeof(uid));
  NCCL_TRY(ctx, api.CommInitRank(&ctx->comm, world_size, uid, rank));
  ctx->world = world_size;
  ctx->rank = rank;
  if (ctx->d_gather) { cudaFree(ctx->d_gather); ctx->d_gather = nullptr; }
  CUDA_TRY(ctx, cudaMalloc(&ctx->d_gather, (size_t)world_size * ctx->lim.max_bands * sizeof(double)));
  return TEBGPU_OK;
}

int32_t tebgpu_comm_destroy(tebgpu_ctx* ctx) {
  if (!ctx) return TEBGPU_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->comm) { nccl_api().CommDestroy(ctx->comm); ctx->comm = nullptr; }
  ctx->world = 1; ctx->rank = 0;
  return TEBGPU_OK;
}

int32_t tebgpu_gather_costs(tebgpu_ctx* ctx, const double* cost_local, int32_t count_local, double* cost_all, int32_t device_ptrs,
                            void* cuda_stream) {
  if (!ctx || !cost_local || !cost_all || count_local < 1) return TEBGPU_ERR_INVALID_ARG;
  CUDA_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = (device_ptrs && cuda_stream) ? (cudaStream_t)cuda_stream : ctx->stream;
  const size_t bytes = (size_t)count_local * sizeof(double);
  if (!ctx->comm) { /* one rank: the gathered vector is the local one */
    if (device_ptrs) { if (cost_all != cost_local) CUDA_TRY(ctx, cudaMemcpyAsync(cost_all, cost_local, bytes, cudaMemcpyDeviceToDevice, st)); }
    else std::memmove(cost_all, cost_local, bytes);
    return TEBGPU_OK;
  }
  if (device_ptrs) {
    NCCL_TRY(ctx, nccl_api().AllGather(cost_local, cost_all, (size_t)count_local, ncclDouble, ctx->comm, st));
    return TEBGPU_OK;
  }
  if (count_local > ctx->lim.max_bands) { ctx->err = "gather of more than max_bands costs"; return TEBGPU_ERR_CAPACITY; }
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_cost, cost_local, bytes, cudaMemcpyHostToDevice, st));
  NCCL_TRY(ctx, nccl_api().AllGather(ctx->d_cost, ctx->d_gather, (size_t)count_local, ncclDouble, ctx->comm, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(cost_all, ctx->d_gather, bytes * ctx->world, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return TEBGPU_OK;
}

int32_t tebgpu_optimize_batch_gather(tebgpu_ctx* ctx, const TebBatch* bt, const TebOptimizeArgs* args, double* cost_all) {
  if (!ctx || !bt || !cost_all || !bt->cost) return TEBGPU_ERR_INVALID_ARG;
  /* the device-side costs of the host entry point live in d_cost: gather them before they travel to the host */
  int32_t rc = tebgpu_optimize_batch(ctx, bt, args);
  if (rc) return rc;
  if (!ctx->comm) { std::memcpy(cost_all, bt->cost, (size_t)bt->B * sizeof(double)); return TEBGPU_OK; }
  cudaStream_t st = ctx->stream;
  NCCL_TRY(ctx, nccl_api().AllGather(ctx->d_cost, ctx->d_gather, (size_t)bt->B, ncclDouble, ctx->comm, st));
  CUDA_TRY(ctx, cudaMemcpyAsync(cost_all, ctx->d_gather, (size_t)bt->B * ctx->world * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(ctx, cudaStreamSynchronize(st));
  return TEBGPU_OK;
}

int32_t tebgpu_select_best(const double* cost, int32_t count, int32_t last_best, int32_t initial_plan,
                           double selection_cost_hysteresis, double selection_prefer_initial_plan) {
  /* HomotopyClassPlanner::selectBestTeb homotopy_class_planner.cpp:564-616 */
  if (!cost || count <= 0) return -1;
  double min_cost = 1.7976931348623157e308;
  int best = -1;
  for (int i = 0; i < count; ++i) {
    double teb_cost;
    if (i == last_best) teb_cost = cost[i] * selection_cost_hysteresis;
    else if (i == initial_plan) teb_cost = cost[i] * selection_prefer_initial_plan;
    else teb_cost = cost[i];
    if (teb_cost < min_cost) { best = i; min_cost = teb_cost; }
  }
  return best;
}

int32_t tebgpu_auto_resize_host(double* rec, int32_t n, int32_t n_cap, double dt_ref, double dt_hysteresis,
                                int32_t min_samples, int32_t max_samples, int32_t fast_mode) {
  if (!rec || n < 1 || n > n_cap) return TEBGPU_ERR_INVALID_ARG;
  int nn = teb_auto_resize_records(rec, n, n_cap, dt_ref, dt_hysteresis, min_samples, max_samples, fast_mode);
  return nn < 0 ? TEBGPU_ERR_CAPACITY : nn;
}

}  /* extern "C" */
