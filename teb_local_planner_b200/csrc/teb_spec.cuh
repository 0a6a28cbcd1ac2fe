/*
 * teb_spec.cuh — speculative Levenberg-Marquardt step ("kernel B", solver 2, the default).
 *
 * g2o's LM loop (SURVEY.md App. A.4) retries a rejected step with lambda *= nu, nu *= 2, up to 10 trials. The trial
 * sequence after consecutive rejections is a pure function of (lambda, nu) at the start of the iteration, and every
 * trial solves the SAME linearised system with a different damping. So the next SPEC_K trials are solved and evaluated
 * concurrently and the accept / reject chain is then replayed in order: bit-for-bit the same decisions as the
 * sequential loop, but the dependent chain per LM iteration shrinks from (trials x solve) to one solve for 95 % of the
 * iterations (measured trial histogram: 1:51 %, 2:12 %, 3:17 %, 4:15 %, 5:5 %, 6:0.2 %).
 *
 *   k_solve_tpb   one THREAD per (band, trial): banded LDL^T (half bandwidth 10) with the 11x11 active window held in
 *                 registers (fully unrolled by 11 so every index is static), rows of H streamed from HBM/L2, factor
 *                 rows streamed out, forward substitution fused, back substitution from the streamed factor.
 *                 Replaces LinearSolverCSparse::solve (optimal_planner.cpp:169-172).
 *   k_trial_eval  one CTA per band, one WARP per trial: trial state x [+] dx, trial chi2 by family, computeScale();
 *                 then one thread replays the accept / reject chain in order and the CTA commits the accepted trial
 *                 state from shared memory. Bands whose K trials were all rejected are appended to a compact list;
 *                 the (rare) retry rounds run over that list only.
 */
#pragma once

#include "teb_kernels.cuh"

namespace tebgpu {

constexpr int SPEC_K_MAX = 8;    /* trials solved concurrently per round: 4, 6 or 8 (runtime, SpecBufs::K) */
constexpr int SPEC_CNT_CAP = 1 << 16; /* retry-list counters per call: outer x inner x rounds */
constexpr int RES_STRIDE = 8;    /* per (band, trial): chi parts [4], scale, ok, lambda, unused */
constexpr int SPEC_LISTS = 8;    /* rotating retry-list buffers: round g reads buffer g % SPEC_LISTS, writes (g + 1) % SPEC_LISTS */

struct SpecBufs {
  double* Lf;    /* [B][K][4 n_cap][12] factor rows: 1/d, z, L[j+1..j+10][j] */
  double* dx;    /* [B][K][4 n_cap]     solution of trial k                   */
  double* res;   /* [B][SPEC_K_MAX][RES_STRIDE]: the stride does not depend on the width of a launch (launches of
                    different widths overlap in time)                           */
  int32_t* need; /* [B] band still needs trials in this LM iteration          */
  int32_t* qmax; /* [B] trials consumed in this LM iteration                  */
  int32_t* cnt;  /* [rounds of the call + 1] length of the retry list a round reads (zeroed per call) */
  int32_t* list; /* [SPEC_LISTS][B] bands of the retry lists, buffer g % SPEC_LISTS is read by round g */
  int32_t K;     /* speculation width of this call                            */
  /* Band selection of a ROUND-0 launch (retry rounds always walk list g):
   *   sel_list != NULL  the bands of that list (sel_cnt entries) - the side stream's share of an LM iteration: the bands
   *                     that needed retries in the previous iteration and were linearised there;
   *   else              every band except those with defer[b] == skip_tag (skip_tag 0: every band).
   * Lf / dx above are the scratch of the LAUNCHING stream: main-stream and side-stream launches overlap in time. */
  const int32_t* sel_list;
  const int32_t* sel_cnt;
  const int32_t* defer;
  int32_t skip_tag;
  /* Retry rounds of the throughput regime are launched twice, as k_solve_lat (grid = lat_cap systems) and as
   * k_solve_tpb; the length of the retry list, known only on the device, decides which of the two does the work:
   * lists of up to lat_cap / K bands (the last retry round: a fraction of a percent of the bands) take the latency
   * mapping instead of paying a thread-per-system solve's fixed 0.26 ms. 0: no such choice, the launched kernel works. */
  int32_t lat_cap;
};
__device__ __forceinline__ bool retry_round_takes_lat(const SpecBufs& sp, int round, int g) {
  return round > 0 && sp.lat_cap > 0 && (long long)sp.cnt[g] * sp.K <= sp.lat_cap;
}

/* the band of system slot `slot` in this launch, or -1 */
__device__ __forceinline__ int spec_band(const DevBatch& db, const SpecBufs& sp, int round, int g, int slot) {
  if (round > 0) return slot < sp.cnt[g] ? sp.list[(size_t)(g % SPEC_LISTS) * db.B + slot] : -1;
  if (sp.sel_list) return slot < *sp.sel_cnt ? sp.sel_list[slot] : -1;
  if (slot >= db.B) return -1;
  if (sp.skip_tag != 0 && deferred_since(sp.defer[slot], sp.skip_tag)) return -1;
  return slot;
}

/* Failure contract of the LM linear solve, shared by every mapping of solver 2 (k_solve_tpb, k_solve_warp, k_solve_lat):
 * a factorisation FAILS - res[5] = 0, TEB_STATUS_CHOL_FAILED, and the trial evaluation takes dx = b as
 * LinearSolverCSparse leaves it - iff some pivot d of the LDL^T is not a positive normal number: d <= 0 (CSparse's "not
 * positive definite", cs_chol stops at d <= 0), NaN, infinite, or subnormal (its reciprocal overflows, and the fast
 * reciprocal of k_solve_lat flushes it to zero). Nothing else fails: a non-finite SOLUTION from valid pivots is reported
 * as a success, as CSparse does, and the non-finite chi2 of that trial ends the LM iteration as it does in g2o. */
__device__ __forceinline__ bool pivot_ok(double d) { return d >= 2.2250738585072014e-308 && isfinite(d); }

/* lambda / nu of trial q0 + k given the state before trial q0 (only rejections in between) */
__device__ __forceinline__ void spec_lambda(double& lambda, double& ni, int k) {
  for (int t = 0; t < k; ++t) { lambda *= ni; ni *= 2; }
}

__device__ __forceinline__ double band_lambda_init(const DevBatch& db, int b, int n) {
  const int chunks_used = (n + db.tile - 1) / db.tile;
  double mx = 0;
  for (int c = 0; c < chunks_used; ++c) mx = fmax(mx, db.dmax_parts[(size_t)b * db.chunks + c]);
  return 1e-5 * mx; /* computeLambdaInit: tau * max diagonal */
}

/* ------------------------------------------------------------------ k_solve_tpb
 * One warp per CTA. Every thread owns a private ring of TPB_RING row slots in shared memory ([slot][16-byte pair][lane]
 * so that a warp access is conflict free) that cp.async (LDGSTS) fills TPB_RING rows ahead of their use: the H rows
 * during the factorisation, the factor rows during the back substitution. No registers are spent on prefetching and
 * the global latency is off the dependent chain. 10 slots (30 KB) instead of 11 let SEVEN solver warps share an SM
 * (7 x 31 KB <= 227 KB; 254 registers x 32 x 7 fits the register file), which is what makes 8192 bands x 4 trials a
 * single wave on 148 SMs. */
constexpr int TPB_RING_MIN = 10;
__host__ __device__ constexpr int tpb_ring_bytes(int ring) { return ring * 6 * 32 * 16; }

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int NPEND>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(NPEND) : "memory"); }

/* TPB_RING = prefetch distance in rows = slots of the private ring: 10 rows (30 KB per warp, 7 warps per SM) is the
 * default; 20 / 30 exist for experiments (TEBGPU_RING) and measured slower - see profiles/r2_history.md. */
template <int TPB_RING>
__global__ void __launch_bounds__(32) k_solve_tpb(DevBatch db, SpecBufs sp, int iteration, int round, int g) {
  extern __shared__ __align__(16) unsigned char ring_raw[];
  const int lane = threadIdx.x;
  const int t = blockIdx.x * 32 + lane;
  const int SPEC_K = sp.K;
  /* system t = K * slot + k; round 0: slot = band, retry rounds: slot indexes the compact list of round g */
  const int slot = t / SPEC_K;
  const int k = t - slot * SPEC_K;
  if (retry_round_takes_lat(sp, round, g)) return; /* k_solve_lat does this round */
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return; /* threads are independent: no warp-level primitive below */
  bool work = true;
  const BandState* st = &db.state[b];
  if (!st->active) work = false;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  if (q0 + k >= 10) work = false;
  if (!work) return;
  const int n = db.n[b];
  const int N = 4 * n;
  double lambda, ni;
  if (round == 0 && iteration == 0) { lambda = band_lambda_init(db, b, n); ni = 2; }
  else { lambda = st->lambda; ni = st->ni; }
  spec_lambda(lambda, ni, k);

  const double* gH = db.Hb + (size_t)b * 4 * db.n_cap * HROW;
  /* factor and solution live in warp-interleaved scratch ([row][16-byte pair][lane] / [row][lane]) so that the 32
   * threads of a warp - 32 different (band, trial) systems - store and load contiguous 512 / 256 byte runs */
  double2* gL = reinterpret_cast<double2*>(sp.Lf + (size_t)blockIdx.x * 32 * 4 * db.n_cap * HROW) + lane;
  double* gx = sp.dx + (size_t)blockIdx.x * 32 * 4 * db.n_cap + lane;
  double* res = sp.res + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;
  const uint32_t ring = smem_u32(ring_raw) + (uint32_t)lane * 16u;                 /* + (slot*6 + pair)*512 */
  const double2* ringp = reinterpret_cast<const double2*>(ring_raw) + lane;       /* [(slot*6 + pair)*32]  */

  /* E[k][m]: H[r][r-k] of the window row r with r % 11 == m; Y[m]: its right-hand side */
  double E[11][11], Y[11];
  /* prologue: rows 0..10 straight into the window, rows 11..21 into the ring */
#pragma unroll
  for (int m = 0; m < 11; ++m) {
    const double2* src = reinterpret_cast<const double2*>(gH + (size_t)m * HROW); /* N >= 12 */
    double h[12];
#pragma unroll
    for (int v = 0; v < 6; ++v) { const double2 d2 = __ldg(src + v); h[2 * v] = d2.x; h[2 * v + 1] = d2.y; }
    if (row_is_real(m, n)) h[0] += lambda;
#pragma unroll
    for (int kk = 0; kk < 11; ++kk) E[kk][m] = (kk <= m) ? h[kk] : 0.0;
    Y[m] = h[11];
  }
#pragma unroll
  for (int m = 0; m < TPB_RING; ++m) {
    const int r = 11 + m;
    if (r < N) {
#pragma unroll
      for (int v = 0; v < 6; ++v) cp_async16(ring + (uint32_t)((m * 6 + v) * 512), gH + (size_t)r * HROW + 2 * v);
    }
    cp_async_commit();
  }
  bool ok = true;
  int rs = 0; /* ring slot that holds row j + 11 */
  /* rows N .. Npad-1 are identity rows: every block of 11 pivots runs unconditionally, which keeps the register
   * window's liveness static (a data-dependent early exit makes the compiler keep all 121 slots alive) */
  for (int j0 = 0; j0 < N; j0 += 11) {
#pragma unroll
    for (int s = 0; s < 11; ++s) {
      const int j = j0 + s;
      const double d = E[0][s];
      if (!pivot_ok(d)) ok = false;
      const double inv = 1.0 / d;
      const double yj = Y[s];
      double cu[11];
#pragma unroll
      for (int u = 1; u <= 10; ++u) cu[u] = E[u][(s + u) % 11];
      const bool live = j < N;
      double2* dst = gL + (size_t)j * 6 * 32; /* pair v at dst[v * 32] */
      if (live) dst[0] = make_double2(inv, yj * inv);
      double lprev = 0;
#pragma unroll
      for (int u = 1; u <= 10; ++u) {
        const double lu = cu[u] * inv;
#pragma unroll
        for (int q = 1; q <= u; ++q) E[u - q][(s + u) % 11] -= lu * cu[q];
        Y[(s + u) % 11] -= lu * yj;
        /* factor row j: 1/d, z_j, L[j+1..j+10][j] */
        if (u & 1) lprev = lu;
        else if (live) dst[(u / 2) * 32] = make_double2(lprev, lu);
      }
      /* install row j + 11 (copied into ring slot rs TPB_RING pivots ago), then refill the slot with row j + 11 + TPB_RING */
      cp_async_wait<TPB_RING - 1>();
      const int rn = j + 11;
      if (rn < N) {
#pragma unroll
        for (int v = 0; v < 5; ++v) { const double2 d2 = ringp[(rs * 6 + v) * 32]; E[2 * v][s] = d2.x; E[2 * v + 1][s] = d2.y; }
        const double2 d2 = ringp[(rs * 6 + 5) * 32];
        E[10][s] = d2.x;
        Y[s] = d2.y;
        if (row_is_real(rn, n)) E[0][s] += lambda;
      } else {
#pragma unroll
        for (int kk = 1; kk < 11; ++kk) E[kk][s] = 0.0;
        E[0][s] = 1.0;
        Y[s] = 0.0;
      }
      if (rn + TPB_RING < N) {
#pragma unroll
        for (int v = 0; v < 6; ++v) cp_async16(ring + (uint32_t)((rs * 6 + v) * 512), gH + (size_t)(rn + TPB_RING) * HROW + 2 * v);
      }
      cp_async_commit();
      rs = (rs + 1 == TPB_RING) ? 0 : rs + 1;
    }
  }
  cp_async_wait<0>();
  res[5] = ok ? 1.0 : 0.0;
  res[6] = lambda;
  if (!ok) return; /* CSparse failure: k_trial_eval uses dx = b */

  /* back substitution x_j = z_j - sum_u L[j+u][j] x_{j+u}; X[m]: x of the row with r % 11 == m.
   * The factor rows written above are read back through the same cp.async ring, 11 rows ahead. */
  double X[11];
#pragma unroll
  for (int m = 0; m < 11; ++m) X[m] = 0;
  const int jtop = ((N - 1) / 11) * 11;
#pragma unroll
  for (int c = 0; c < TPB_RING; ++c) { /* rows jtop + 10 - c, c = 0 .. TPB_RING - 1 */
    const int j = jtop + 10 - c;
    if (j < N) {
#pragma unroll
      for (int v = 0; v < 6; ++v) cp_async16(ring + (uint32_t)((c * 6 + v) * 512), gL + ((size_t)j * 6 + v) * 32);
    }
    cp_async_commit();
  }
  rs = 0;
  for (int j0 = jtop; j0 >= 0; j0 -= 11) {
#pragma unroll
    for (int s = 10; s >= 0; --s) {
      const int j = j0 + s;
      const bool live = j < N;
      cp_async_wait<TPB_RING - 1>();
      double l[12];
      if (live) {
#pragma unroll
        for (int v = 0; v < 6; ++v) { const double2 d2 = ringp[(rs * 6 + v) * 32]; l[2 * v] = d2.x; l[2 * v + 1] = d2.y; }
      } else {
#pragma unroll
        for (int v = 0; v < 12; ++v) l[v] = 0.0;
      }
      if (j - TPB_RING >= 0) {
#pragma unroll
        for (int v = 0; v < 6; ++v) cp_async16(ring + (uint32_t)((rs * 6 + v) * 512), gL + ((size_t)(j - TPB_RING) * 6 + v) * 32);
      }
      cp_async_commit();
      rs = (rs + 1 == TPB_RING) ? 0 : rs + 1;
      double acc = l[1];
#pragma unroll
      for (int u = 10; u >= 1; --u) acc -= l[1 + u] * X[(s + u) % 11];
      X[s] = acc;
      if (live) gx[(size_t)j * 32] = acc;
    }
  }
  cp_async_wait<0>();
}

/* Accept / reject replay (OptimizationAlgorithmLevenberg::solve, SURVEY App. A.4), sequential over the K trials of one
 * band; run by one thread. Returns the accepted trial (or -1). */
struct DecideArgs { /* passed by value: a reference to the kernel parameters would force them into local memory */
  BandState* st;
  const double* chi_parts; /* this band's tile partials */
  double lambda_init;
  int32_t* need;           /* &need[b] */
  int32_t* qmax;           /* &qmax[b] */
  int32_t* cnt_next;       /* &cnt[g + 1] */
  int32_t* list_next;      /* list buffer of round g + 1 */
  int32_t* defer;          /* &defer[b] */
  int32_t tag;             /* inner-iteration tag written to defer[b] when the band is queued */
  int32_t b, n, K, iteration, round, q0;
  int32_t tile;            /* poses per kernel-A tile */
};
__device__ __forceinline__ int spec_decide(const DecideArgs a, const double* sRes) {
  const int SPEC_K = a.K, n = a.n, round = a.round, iteration = a.iteration, q0 = a.q0;
  BandState* st = a.st;
  int accepted = -1;
  double lambda, ni, currentChi;
  double cur_parts[4], last_parts[4];
  int q;
  if (round == 0) {
    /* chi2 at the linearisation point = sum of the kernel-A tile partials (computeActiveErrors) */
    const int chunks_used = (n + a.tile - 1) / a.tile;
    const double* cp = a.chi_parts;
    for (int c = 0; c < 4; ++c) cur_parts[c] = 0;
    for (int ch = 0; ch < chunks_used; ++ch)
      for (int c = 0; c < 4; ++c) cur_parts[c] += cp[4 * ch + c];
    currentChi = cur_parts[0] + cur_parts[1] + cur_parts[2] + cur_parts[3];
    if (iteration == 0) { lambda = a.lambda_init; ni = 2; }
    else { lambda = st->lambda; ni = st->ni; }
    q = 0;
  } else {
    lambda = st->lambda; ni = st->ni; currentChi = st->current_chi; q = q0;
    for (int c = 0; c < 4; ++c) cur_parts[c] = st->parts_cur[c];
  }
  for (int c = 0; c < 4; ++c) last_parts[c] = st->parts_last[c];
  int status_add = 0;
  bool done = false;
  double rho = 0;
  for (int kk = 0; kk < SPEC_K && q < 10; ++kk) {
    const double* r = sRes + kk * RES_STRIDE;
    const bool ok2 = r[5] != 0.0;
    for (int c = 0; c < 4; ++c) last_parts[c] = r[c];
    double tempChi = r[0] + r[1] + r[2] + r[3];
    if (!ok2) { tempChi = 1.7976931348623157e308; status_add |= TEB_STATUS_CHOL_FAILED; }
    const double scale = r[4] + 1e-3;
    rho = (currentChi - tempChi) / scale;
    if (rho > 0 && isfinite(tempChi)) {
      const double t3 = 2 * rho - 1;
      double alpha = 1. - t3 * t3 * t3; /* pow(2 rho - 1, 3) to within 1.5 ulp, no libm call on the replay path */
      alpha = fmin(alpha, 2. / 3.);
      const double scaleFactor = fmax(1. / 3., alpha);
      lambda *= scaleFactor;
      ni = 2;
      currentChi = tempChi;
      for (int c = 0; c < 4; ++c) cur_parts[c] = last_parts[c];
      accepted = kk;
    } else {
      lambda *= ni;
      ni *= 2;
      if (!isfinite(lambda)) { status_add |= TEB_STATUS_NONFINITE; done = true; break; }
    }
    q++;
    if (!(rho < 0 && q < 10)) { done = true; break; }
  }
  st->lambda = lambda;
  st->ni = ni;
  st->current_chi = currentChi;
  st->chi2_final = currentChi;
  for (int c = 0; c < 4; ++c) { st->parts_last[c] = last_parts[c]; st->parts_cur[c] = cur_parts[c]; }
  *a.qmax = q;
  int stt = st->status | status_add;
  if (done) {
    const bool terminate = (q == 10 || rho == 0 || !isfinite(lambda));
    st->lm_iters += 1;
    if (terminate) { stt |= TEB_STATUS_TERMINATED; st->active = 0; }
    else stt &= ~TEB_STATUS_TERMINATED;
    *a.need = 0;
  } else {
    /* all K trials rejected: queue the band for the next round (slot order is arbitrary, results do not depend
     * on it: every band only touches its own data) */
    *a.need = 1;
    const int s2 = atomicAdd(a.cnt_next, 1);
    a.list_next[s2] = a.b;
    *a.defer = a.tag;
  }
  st->status = stt;
  return accepted;
}

/* ------------------------------------------------------------------ k_trial_eval: CTA per band, warp k = trial k.
 * The K trial solutions of a band sit in adjacent lanes of the solver's interleaved scratch (one 32-byte sector per
 * row at K = 4), so the CTA stages them - and the scene's obstacle table and the K trial states - in shared memory
 * once. After the K chi2 are known, thread 0 replays g2o's accept / reject chain (SURVEY App. A.4) in trial order and
 * the CTA copies the accepted trial state (discardTop()) from shared memory into the band. */
__host__ __device__ inline size_t eval_smem_bytes(int n_cap, int M_cap, int K) {
  return ((size_t)K * 2 + 2) * 4 * n_cap * sizeof(double) + (size_t)(M_cap > 0 ? M_cap : 1) * sizeof(TebObstacle) +
         (size_t)K * RES_STRIDE * sizeof(double) + 32;
}

template <int MINB, bool GEOM>
__global__ void __launch_bounds__(32 * SPEC_K_MAX, MINB) k_trial_eval(DevBatch db, KParams kp, SpecBufs sp, int iteration,
                                                                int round, int g, int tag) {
  extern __shared__ __align__(16) unsigned char ev_raw[];
  const int SPEC_K = sp.K;
  const int slot = blockIdx.x;
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return;
  const int tid = threadIdx.x, lane = tid & 31, k = tid >> 5;
  BandState* st = &db.state[b];
  if (!st->active) return;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  const int n = db.n[b];
  const int N = 4 * n;
  double* sdx = reinterpret_cast<double*>(ev_raw);           /* [K][4 n_cap] */
  double* sT = sdx + (size_t)SPEC_K * 4 * db.n_cap;           /* [K][n_cap][4] */
  double* sP0 = sT + (size_t)SPEC_K * 4 * db.n_cap;           /* [n_cap][4] current band */
  double* sB = sP0 + (size_t)4 * db.n_cap;                    /* [4 n_cap] right-hand side */
  double* sRes = sB + (size_t)4 * db.n_cap;                   /* [K][RES_STRIDE] */
  int* sAcc = reinterpret_cast<int*>(sRes + (size_t)SPEC_K * RES_STRIDE);
  TebObstacle* so = reinterpret_cast<TebObstacle*>(sAcc + 4);
  const int sc = db.scene_id[b];
  const int M = db.obst_count[sc];
  {
    const TebObstacle* go = db.obstacles + (size_t)sc * db.M_cap;
    for (int m = tid; m < M; m += 32 * SPEC_K) so[m] = go[m];
    /* rows of the K trial solutions: system index K slot + k -> solver warp (K slot + k) >> 5, lane (K slot + k) & 31:
     * the trials of a band are adjacent lanes of the interleaved scratch (K even: pairs never straddle a tile) */
    const double* gP = db.poses + (size_t)b * db.n_cap * 4;
    const double* grhs = db.rhs + (size_t)b * 4 * db.n_cap;
    for (int r = tid; r < N; r += 32 * SPEC_K) {
      sP0[r] = gP[r];
      sB[r] = grhs[r];
      for (int kk = 0; kk < SPEC_K; kk += 2) {
        const int tsys = slot * SPEC_K + kk;
        const double2 a = *reinterpret_cast<const double2*>(sp.dx + (size_t)(tsys >> 5) * 32 * 4 * db.n_cap +
                                                            (size_t)r * 32 + (tsys & 31));
        sdx[(size_t)kk * 4 * db.n_cap + r] = a.x;
        sdx[(size_t)(kk + 1) * 4 * db.n_cap + r] = a.y;
      }
    }
  }
  __syncthreads();
  const bool mine = (q0 + k < 10);
  const double* res = sp.res + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;
  double chi[4] = {0, 0, 0, 0};
  double scl = 0;
  bool ok = true;
  if (mine) {
    ok = res[5] != 0.0;
    const double lambda = res[6];
    const double* mydx = sdx + (size_t)k * 4 * db.n_cap;
    double* myT = sT + (size_t)k * 4 * db.n_cap;
    /* trial state x [+] dx and computeScale() = sum dx (lambda dx + b) */
    for (int r = lane; r < N; r += 32) {
      double xv = sP0[r];
      if (row_is_real(r, n)) {
        const double bb = sB[r];
        const double dx = ok ? mydx[r] : bb; /* CSparse leaves x = b when the factorisation fails */
        scl += dx * (lambda * dx + bb);
        xv = ((r & 3) == 2) ? normalize_theta(xv + dx) : xv + dx;
      }
      myT[r] = xv;
    }
    __syncwarp();
    const double* vs = db.vel_start + 4 * (size_t)b;
    const double* vg = db.vel_goal + 4 * (size_t)b;
    /* contiguous chunk per lane: sin/cos and segment velocities are carried from pose to pose */
    const int per = (n + 31) >> 5;
    const int i0 = lane * per, i1 = min(i0 + per, n);
    ChainCarry cy;
    cy.has_cs = false; cy.has_seg = false;
    for (int i = i0; i < i1; ++i) pose_chi2<GEOM>(kp, db, b, sc, i, n, myT, so, M, vs, vg, chi, cy);
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) chi[c] = warp_sum(chi[c]);
  scl = warp_sum(scl);
  if (mine && lane == 0) {
    double* r = sRes + k * RES_STRIDE;
    r[0] = chi[0]; r[1] = chi[1]; r[2] = chi[2]; r[3] = chi[3];
    r[4] = scl;
    r[5] = ok ? 1.0 : 0.0;
  }
  __syncthreads();

  /* ---- accept / reject replay, sequential over the K trials */
  if (tid == 0) {
    DecideArgs da;
    da.st = st; da.chi_parts = db.chi_parts + (size_t)b * db.chunks * 4;
    da.lambda_init = (round == 0 && iteration == 0) ? band_lambda_init(db, b, n) : 0.0;
    da.need = sp.need + b; da.qmax = sp.qmax + b; da.cnt_next = sp.cnt + g + 1;
    da.list_next = sp.list + (size_t)((g + 1) % SPEC_LISTS) * db.B;
    da.defer = db.defer + b; da.tag = tag;
    da.b = b; da.n = n; da.K = SPEC_K; da.iteration = iteration; da.round = round; da.q0 = q0; da.tile = db.tile;
    const int accepted = spec_decide(da, sRes);
    sAcc[0] = accepted;
  }
  __syncthreads();
  const int accepted = sAcc[0];
  if (accepted >= 0) { /* discardTop(): the accepted trial state becomes the band */
    double* gP = db.poses + (size_t)b * db.n_cap * 4;
    const double* aT = sT + (size_t)accepted * 4 * db.n_cap;
    for (int r = tid; r < N; r += 32 * SPEC_K) gP[r] = aT[r];
  }
}


/* ====================================================================================================================
 * k_trial_eval2 — trial evaluation, second generation (the default): ONE LANE PER POSE.
 * A CTA still owns one band and stages the current band, the K trial solutions, the right-hand side and the scene's
 * obstacle table once; but the chi2 of a trial is no longer a per-lane walk over a chunk of poses with a dependent carry:
 * a warp takes a (trial, 30-pose tile) task, every lane forms the trial state of its own pose (x [+] dx), its sin / cos
 * and the velocities of its own segment, the right neighbour's values arrive by warp shuffles (2 halo lanes per tile),
 * and the lane evaluates all cost terms anchored at its pose. Tile partials are folded in a fixed order, then one thread
 * replays g2o's accept / reject chain (spec_decide) and the CTA commits the accepted trial state.
 * ==================================================================================================================== */
constexpr int EV2_THREADS = 256;
constexpr int EV2_MINB = 4;       /* CTAs per SM the throughput variant is compiled for (register cap 85) */
constexpr int EV2_TILE = 30;      /* poses evaluated per warp task: lanes 0 .. 29 (lanes 30, 31: halo) */
__host__ __device__ inline int ev2_tiles(int n_cap) { return (n_cap + EV2_TILE - 1) / EV2_TILE; }
__host__ __device__ inline size_t eval2_smem_bytes(int n_cap, int M_cap, int K) {
  return ((size_t)K + 2) * 4 * n_cap * sizeof(double) + (size_t)(M_cap > 0 ? M_cap : 1) * sizeof(TebObstacle) +
         ((size_t)K * ev2_tiles(n_cap) * 5 + (size_t)K * RES_STRIDE) * sizeof(double) + 64;
}

/* chi2 contributions of everything anchored at pose i of a trial state held in registers: chain edges of segment i,
 * time-optimal edge i, unary edges of pose i. (xa .. dta, ca, sa): pose i; (xb .. dtb, cb, sb): pose i+1; s1 / s2:
 * velocities of the segments i and i+1. Same arithmetic as pose_chi2 (teb_kernels.cuh). */
template <bool GEOM>
__device__ __forceinline__ void pose_chi2_lane(const KParams& kp, const DevBatch& db, int b, int sc, int i, int n, double xa,
                                               double ya, double tha, double dta, double ca, double sa, double xb, double yb,
                                               double thb, double dtb, double cb, double sb, const SegVal& s1, const SegVal& s2,
                                               const TebObstacle* so, int M, const double* vs, const double* vg, double (&chi)[4]) {
  if (i <= n - 2) {
    const double dx = xb - xa, dy = yb - ya;
    double sl, csum = 0;
    if (kp.has_vel && kp.holo_vel) {
      double e[3], s3[3], c0, c1;
      holo_velocity_terms(kp, s1.vx, s1.vy, s1.w, e, s3, c0, c1);
      const double e0 = kp.sw_vel_x * e[0], e1 = kp.sw_vel_y * e[1], e2 = kp.sw_vel_th * e[2];
      csum += e0 * e0 + e1 * e1 + e2 * e2;
    } else if (kp.has_vel) {
      const double e0 = kp.sw_vel_x * pen_interval2(s1.v, -kp.p.max_vel_x_backwards, kp.p.max_vel_x, kp.p.penalty_epsilon, sl);
      const double e1 = kp.sw_vel_th * pen_interval(s1.w, kp.p.max_vel_theta, kp.p.penalty_epsilon, sl);
      csum += e0 * e0 + e1 * e1;
    }
    if (kp.has_kin) {
      const double e0 = kp.sw_kin_nh * fabs((ca + cb) * dy - (sa + sb) * dx);
      double e1 = 0;
      if (!kp.carlike) {
        e1 = pen_below(dx * ca + dy * sa, 0, 0, sl);
      } else {
        const double ad = normalize_theta(thb - tha);
        if (ad != 0) {
          const double nrm = sqrt(dx * dx + dy * dy);
          const double r = kp.p.exact_arc_length ? fabs(nrm / (2 * sin(ad / 2))) : nrm / fabs(ad);
          e1 = pen_below(r, kp.p.min_turning_radius, 0.0, sl);
        }
      }
      e1 *= kp.sw_kin_2;
      csum += e0 * e0 + e1 * e1;
    }
    if (kp.has_sp) {
      const double e = kp.sw_sp * sqrt(dx * dx + dy * dy);
      csum += e * e;
    }
    if (kp.has_rot && i < 3) {
      const int rd = db.prefer_rotdir ? db.prefer_rotdir[b] : 0;
      if (rd == TEB_ROTDIR_LEFT || rd == TEB_ROTDIR_RIGHT) {
        const double meas = (rd == TEB_ROTDIR_LEFT) ? 1.0 : -1.0;
        const double e = kp.sw_rot * pen_below(meas * normalize_theta(thb - tha), 0, 0, sl);
        csum += e * e;
      }
    }
    if (kp.has_acc && kp.holo_acc) {
      const double idt1 = 1.0 / dta;
      const double lim[3] = {kp.p.acc_lim_x, kp.p.acc_lim_y, kp.p.acc_lim_theta};
      const double sw[3] = {kp.sw_acc_x, kp.sw_acc_y, kp.sw_acc_th};
      const double u1[3] = {s1.vx, s1.vy, s1.w};
      if (i <= n - 3) {
        const double iT = 1.0 / (dta + dtb);
        const double u2[3] = {s2.vx, s2.vy, s2.w};
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double e = sw[r] * pen_interval((u2[r] - u1[r]) * 2 * iT, lim[r], kp.p.penalty_epsilon, sl);
          csum += e * e;
        }
      } else if (vg[3] != 0) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double e = sw[r] * pen_interval((vg[r] - u1[r]) * idt1, lim[r], kp.p.penalty_epsilon, sl);
          csum += e * e;
        }
      }
      if (i == 0 && vs[3] != 0) {
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const double e = sw[r] * pen_interval((u1[r] - vs[r]) * idt1, lim[r], kp.p.penalty_epsilon, sl);
          csum += e * e;
        }
      }
    } else if (kp.has_acc) {
      const double idt1 = 1.0 / dta;
      if (i <= n - 3) {
        const double iT = 1.0 / (dta + dtb);
        const double e0 = kp.sw_acc_x * pen_interval((s2.v - s1.v) * 2 * iT, kp.p.acc_lim_x, kp.p.penalty_epsilon, sl);
        const double e1 = kp.sw_acc_th * pen_interval((s2.w - s1.w) * 2 * iT, kp.p.acc_lim_theta, kp.p.penalty_epsilon, sl);
        csum += e0 * e0 + e1 * e1;
      } else if (vg[3] != 0) {
        const double e0 = kp.sw_acc_x * pen_interval((vg[0] - s1.v) * idt1, kp.p.acc_lim_x, kp.p.penalty_epsilon, sl);
        const double e1 = kp.sw_acc_th * pen_interval((vg[2] - s1.w) * idt1, kp.p.acc_lim_theta, kp.p.penalty_epsilon, sl);
        csum += e0 * e0 + e1 * e1;
      }
      if (i == 0 && vs[3] != 0) {
        const double e0 = kp.sw_acc_x * pen_interval((s1.v - vs[0]) * idt1, kp.p.acc_lim_x, kp.p.penalty_epsilon, sl);
        const double e1 = kp.sw_acc_th * pen_interval((s1.w - vs[2]) * idt1, kp.p.acc_lim_theta, kp.p.penalty_epsilon, sl);
        csum += e0 * e0 + e1 * e1;
      }
    }
    if (kp.has_vor) { /* EdgeVelocityObstacleRatio: obstacles associated with pose i (pose 0 included) */
      const unsigned long long* am = db.assoc + ((size_t)b * db.n_cap + i) * db.MW;
      for (int w = 0; w < db.MW; ++w) {
        unsigned long long mask = am[w];
        while (mask) {
          const int m = (w << 6) + __ffsll((long long)mask) - 1;
          mask &= mask - 1;
          const TebObstacle ob = so[m];
          double dratio;
          const double d = robot_obstacle_distance_only<GEOM>(kp, db.obst_vertices + (size_t)sc * db.PV_cap * 2, xa, ya, ca, sa, ob,
                                                        ob.x, ob.y, 0.0, 0.0);
          const double ratio = proximity_ratio(kp, d, dratio);
          const double e0 = pen_interval(s1.v, ratio * kp.p.max_vel_x, 0, sl);
          const double e1 = pen_interval(s1.w, ratio * kp.p.max_vel_theta, 0, sl);
          csum += kp.p.weight_velocity_obstacle_ratio * (e0 * e0 + e1 * e1);
        }
      }
    }
    chi[3] += csum;
    if (kp.has_time) chi[2] += kp.p.weight_optimaltime * dta * dta;
  }
  double U[6], ub[3];
  unary_terms<GEOM>(kp, db, b, sc, i, n, xa, ya, ca, sa, so, M, false, U, ub, chi[0], chi[1]);
}

/* One (trial, 30-pose tile) task of a warp: lane -> pose i = tile * 30 + lane (lanes 30, 31 are the halo). Forms the trial
 * state x [+] dx of its pose, gets the right neighbour's by shuffles, evaluates every cost term anchored at the pose and
 * returns the warp sums: chi2 by family and the computeScale() part of the owned rows. Shared by k_trial_eval2 / 3. */
template <bool GEOM>
__device__ __forceinline__ void eval_tile_task(const KParams& kp, const DevBatch& db, int b, int sc, int n, int tile, int lane, bool ok,
                                               double lambda, const double* mydx, const double* sP0, const double* sB,
                                               const TebObstacle* so, int M, const double* vs, const double* vg, double (&chi)[4],
                                               double& scl) {
  const int i = tile * EV2_TILE + lane;
  chi[0] = chi[1] = chi[2] = chi[3] = 0;
  scl = 0;
  double x = 0, y = 0, th = 0, dt = 1, ca = 1, sa = 0;
  SegVal s1;
  s1.v = 0; s1.w = 0; s1.vx = 0; s1.vy = 0;
  const bool have = i < n;
  const bool own = have && lane < EV2_TILE;
  if (have) { /* trial state x [+] dx (VertexPose::oplusImpl / VertexTimeDiff::oplusImpl), computeScale() on the owned rows */
    double v[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int r = 4 * i + c;
      double xv = sP0[r];
      if (row_is_real(r, n)) {
        const double bb = sB[r];
        const double dxv = ok ? mydx[r] : bb; /* CSparse leaves x = b when the factorisation fails */
        if (own) scl += dxv * (lambda * dxv + bb);
        xv = (c == 2) ? normalize_theta(xv + dxv) : xv + dxv;
      }
      v[c] = xv;
    }
    x = v[0]; y = v[1]; th = v[2]; dt = v[3];
    sincos(th, &sa, &ca);
  }
  /* pose i+1 from the right neighbour */
  const double xb = __shfl_down_sync(0xffffffffu, x, 1), yb = __shfl_down_sync(0xffffffffu, y, 1);
  const double thb = __shfl_down_sync(0xffffffffu, th, 1), dtb = __shfl_down_sync(0xffffffffu, dt, 1);
  const double cb = __shfl_down_sync(0xffffffffu, ca, 1), sb = __shfl_down_sync(0xffffffffu, sa, 1);
  if (have && i <= n - 2 && lane < 31) s1 = seg_value(kp, x, y, th, ca, sa, xb, yb, thb, dt);
  SegVal s2;
  s2.v = __shfl_down_sync(0xffffffffu, s1.v, 1); s2.w = __shfl_down_sync(0xffffffffu, s1.w, 1);
  s2.vx = __shfl_down_sync(0xffffffffu, s1.vx, 1); s2.vy = __shfl_down_sync(0xffffffffu, s1.vy, 1);
  if (own) pose_chi2_lane<GEOM>(kp, db, b, sc, i, n, x, y, th, dt, ca, sa, xb, yb, thb, dtb, cb, sb, s1, s2, so, M, vs, vg, chi);
#pragma unroll
  for (int c = 0; c < 4; ++c) chi[c] = warp_sum(chi[c]);
  scl = warp_sum(scl);
}

template <bool GEOM, int NT> /* NT = 256 (throughput regime, 2 CTAs per SM) or 512 (latency regime: more warps per band) */
__global__ void __launch_bounds__(NT, NT == 256 ? (GEOM ? 2 : EV2_MINB) : 1) k_trial_eval2(const __grid_constant__ DevBatch db, const __grid_constant__ KParams kp,
                                                             const __grid_constant__ SpecBufs sp, int iteration, int round,
                                                             int g, int tag) {
  extern __shared__ __align__(16) unsigned char ev_raw[];
  const int SPEC_K = sp.K;
  const int slot = blockIdx.x;
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthreads = blockDim.x; /* <= NT: as many warps as the band has 30-pose tiles, so that the K x tiles tasks split evenly */
  BandState* st = &db.state[b];
  if (!st->active) return;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  const int n = db.n[b];
  const int N = 4 * n;
  const int tiles = (n + EV2_TILE - 1) / EV2_TILE;
  double* sdx = reinterpret_cast<double*>(ev_raw);            /* [K][4 n_cap] trial solutions */
  double* sP0 = sdx + (size_t)SPEC_K * 4 * db.n_cap;           /* [n_cap][4] current band */
  double* sB = sP0 + (size_t)4 * db.n_cap;                     /* [4 n_cap] right-hand side */
  double* sPart = sB + (size_t)4 * db.n_cap;                   /* [K][tiles(n_cap)][5] tile partials: chi by family, scale */
  double* sRes = sPart + (size_t)SPEC_K * ev2_tiles(db.n_cap) * 5; /* [K][RES_STRIDE] */
  int* sAcc = reinterpret_cast<int*>(sRes + (size_t)SPEC_K * RES_STRIDE);
  TebObstacle* so = reinterpret_cast<TebObstacle*>(sAcc + 4);
  const int sc = db.scene_id[b];
  const int M = db.obst_count[sc];
  {
    const TebObstacle* go = db.obstacles + (size_t)sc * db.M_cap;
    for (int m = tid; m < M; m += nthreads) so[m] = go[m];
    const double* gP = db.poses + (size_t)b * db.n_cap * 4;
    const double* grhs = db.rhs + (size_t)b * 4 * db.n_cap;
    /* the K trial solutions of a band sit in adjacent lanes of the solver's interleaved scratch (K even) */
    for (int r = tid; r < N; r += nthreads) {
      sP0[r] = gP[r];
      sB[r] = grhs[r];
      for (int kk = 0; kk < SPEC_K; kk += 2) {
        const int tsys = slot * SPEC_K + kk;
        const double2 a = *reinterpret_cast<const double2*>(sp.dx + (size_t)(tsys >> 5) * 32 * 4 * db.n_cap + (size_t)r * 32 + (tsys & 31));
        sdx[(size_t)kk * 4 * db.n_cap + r] = a.x;
        sdx[(size_t)(kk + 1) * 4 * db.n_cap + r] = a.y;
      }
    }
  }
  __syncthreads();
  const int kact = min(SPEC_K, 10 - q0); /* trials of this round that exist (g2o stops after 10) */
  const double* vs = db.vel_start + 4 * (size_t)b;
  const double* vg = db.vel_goal + 4 * (size_t)b;
  for (int task = warp; task < kact * tiles; task += nthreads / 32) {
    const int k = task / tiles, tile = task - k * tiles;
    const double* res = sp.res + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;
    double chi[4], scl;
    eval_tile_task<GEOM>(kp, db, b, sc, n, tile, lane, res[5] != 0.0, res[6], sdx + (size_t)k * 4 * db.n_cap, sP0, sB, so, M, vs, vg,
                         chi, scl);
    if (lane == 0) {
      double* pp = sPart + ((size_t)k * ev2_tiles(db.n_cap) + tile) * 5;
      pp[0] = chi[0]; pp[1] = chi[1]; pp[2] = chi[2]; pp[3] = chi[3]; pp[4] = scl;
    }
  }
  __syncthreads();
  if (tid < kact) { /* fold the tile partials of trial tid in tile order */
    double a[5] = {0, 0, 0, 0, 0};
    for (int t = 0; t < tiles; ++t) {
      const double* pp = sPart + ((size_t)tid * ev2_tiles(db.n_cap) + t) * 5;
#pragma unroll
      for (int c = 0; c < 5; ++c) a[c] += pp[c];
    }
    double* r = sRes + tid * RES_STRIDE;
    r[0] = a[0]; r[1] = a[1]; r[2] = a[2]; r[3] = a[3]; r[4] = a[4];
    r[5] = sp.res[((size_t)b * SPEC_K_MAX + tid) * RES_STRIDE + 5];
  }
  __syncthreads();
  /* ---- accept / reject replay, sequential over the K trials */
  if (tid == 0) {
    DecideArgs da;
    da.st = st; da.chi_parts = db.chi_parts + (size_t)b * db.chunks * 4;
    da.lambda_init = (round == 0 && iteration == 0) ? band_lambda_init(db, b, n) : 0.0;
    da.need = sp.need + b; da.qmax = sp.qmax + b; da.cnt_next = sp.cnt + g + 1;
    da.list_next = sp.list + (size_t)((g + 1) % SPEC_LISTS) * db.B;
    da.defer = db.defer + b; da.tag = tag;
    da.b = b; da.n = n; da.K = SPEC_K; da.iteration = iteration; da.round = round; da.q0 = q0; da.tile = db.tile;
    sAcc[0] = spec_decide(da, sRes);
  }
  __syncthreads();
  const int accepted = sAcc[0];
  if (accepted >= 0) { /* discardTop(): the accepted trial state becomes the band (same arithmetic as above) */
    double* gP = db.poses + (size_t)b * db.n_cap * 4;
    const double* adx = sdx + (size_t)accepted * 4 * db.n_cap;
    const bool ok = sRes[accepted * RES_STRIDE + 5] != 0.0;
    for (int r = tid; r < N; r += nthreads) {
      if (!row_is_real(r, n)) continue;
      const double dxv = ok ? adx[r] : sB[r];
      const double xv = sP0[r] + dxv;
      gP[r] = ((r & 3) == 2) ? normalize_theta(xv) : xv;
    }
  }
}

/* ====================================================================================================================
 * k_trial_eval3 — the trial evaluation of the LATENCY regime (one planning request: a few dozen bands). k_trial_eval2
 * gives a band ONE CTA, i.e. 32 candidates keep 32 of the 148 SMs busy for 33 us. Here a CTA owns one (band, trial)
 * pair - grid (K, bands), one warp per 30-pose tile - so a request spreads over the whole chip; the per-trial chi2 /
 * scale go to sp.res in global memory and the LAST CTA of a band to arrive (one atomic counter per band) replays the
 * accept / reject chain and commits the accepted trial, reading its dx back from the solver's scratch.
 * Same tile tasks, same fold order, same spec_decide as k_trial_eval2: the results are bit-identical.
 * ==================================================================================================================== */
__host__ __device__ inline size_t eval3_smem_bytes(int n_cap, int M_cap, int K) {
  return (size_t)3 * 4 * n_cap * sizeof(double) + (size_t)(M_cap > 0 ? M_cap : 1) * sizeof(TebObstacle) +
         ((size_t)ev2_tiles(n_cap) * 5 + (size_t)K * RES_STRIDE) * sizeof(double) + 64;
}

template <bool GEOM>
__global__ void __launch_bounds__(512, 1) k_trial_eval3(const __grid_constant__ DevBatch db, const __grid_constant__ KParams kp,
                                                        const __grid_constant__ SpecBufs sp, int iteration, int round, int g,
                                                        int tag, int32_t* arrive) {
  extern __shared__ __align__(16) unsigned char ev_raw[];
  const int SPEC_K = sp.K;
  const int k = blockIdx.x, slot = blockIdx.y;
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthreads = blockDim.x;
  BandState* st = &db.state[b];
  if (!st->active) return;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  const int kact = min(SPEC_K, 10 - q0); /* trials of this round that exist (g2o stops after 10) */
  if (k >= kact) return;
  const int n = db.n[b];
  const int N = 4 * n;
  const int tiles = (n + EV2_TILE - 1) / EV2_TILE;
  double* sdx = reinterpret_cast<double*>(ev_raw);            /* [4 n_cap] this trial's solution */
  double* sP0 = sdx + (size_t)4 * db.n_cap;                    /* [n_cap][4] current band */
  double* sB = sP0 + (size_t)4 * db.n_cap;                     /* [4 n_cap] right-hand side */
  double* sPart = sB + (size_t)4 * db.n_cap;                   /* [tiles(n_cap)][5] tile partials: chi by family, scale */
  double* sRes = sPart + (size_t)ev2_tiles(db.n_cap) * 5;      /* [K][RES_STRIDE], filled by the deciding CTA */
  int* sAcc = reinterpret_cast<int*>(sRes + (size_t)SPEC_K * RES_STRIDE);
  TebObstacle* so = reinterpret_cast<TebObstacle*>(sAcc + 4);
  const int sc = db.scene_id[b];
  const int M = db.obst_count[sc];
  double* gP = db.poses + (size_t)b * db.n_cap * 4;
  auto dx_of = [&](int kk) { /* trial kk's solution in the solver's interleaved scratch: + r * 32 */
    const int tsys = slot * SPEC_K + kk;
    return sp.dx + (size_t)(tsys >> 5) * 32 * 4 * db.n_cap + (tsys & 31);
  };
  {
    const TebObstacle* go = db.obstacles + (size_t)sc * db.M_cap;
    for (int m = tid; m < M; m += nthreads) so[m] = go[m];
    const double* grhs = db.rhs + (size_t)b * 4 * db.n_cap;
    const double* gdx = dx_of(k);
    for (int r = tid; r < N; r += nthreads) {
      sP0[r] = gP[r];
      sB[r] = grhs[r];
      sdx[r] = gdx[(size_t)r * 32];
    }
  }
  __syncthreads();
  const double* vs = db.vel_start + 4 * (size_t)b;
  const double* vg = db.vel_goal + 4 * (size_t)b;
  double* res = sp.res + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;
  {
    const bool ok = res[5] != 0.0;
    const double lambda = res[6];
    for (int tile = warp; tile < tiles; tile += nthreads / 32) {
      double chi[4], scl;
      eval_tile_task<GEOM>(kp, db, b, sc, n, tile, lane, ok, lambda, sdx, sP0, sB, so, M, vs, vg, chi, scl);
      if (lane == 0) {
        double* pp = sPart + (size_t)tile * 5;
        pp[0] = chi[0]; pp[1] = chi[1]; pp[2] = chi[2]; pp[3] = chi[3]; pp[4] = scl;
      }
    }
  }
  __syncthreads();
  if (tid == 0) { /* fold the tile partials in tile order, publish, arrive */
    double a[5] = {0, 0, 0, 0, 0};
    for (int t = 0; t < tiles; ++t) {
#pragma unroll
      for (int c = 0; c < 5; ++c) a[c] += sPart[(size_t)t * 5 + c];
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) __stcg(res + c, a[c]);
    __threadfence();
    const int old = atomicAdd(arrive + b, 1);
    sAcc[1] = (old == kact - 1);
  }
  __syncthreads();
  if (!sAcc[1]) return;
  /* ---- the last CTA of the band: accept / reject replay, sequential over the K trials */
  __threadfence();
  for (int e = tid; e < kact * RES_STRIDE; e += nthreads) /* L2 reads: the other trials' rows were written by other SMs */
    sRes[e] = __ldcg(sp.res + (size_t)b * SPEC_K_MAX * RES_STRIDE + e);
  __syncthreads();
  if (tid == 0) {
    arrive[b] = 0; /* ready for the next round (stream order) */
    DecideArgs da;
    da.st = st; da.chi_parts = db.chi_parts + (size_t)b * db.chunks * 4;
    da.lambda_init = (round == 0 && iteration == 0) ? band_lambda_init(db, b, n) : 0.0;
    da.need = sp.need + b; da.qmax = sp.qmax + b; da.cnt_next = sp.cnt + g + 1;
    da.list_next = sp.list + (size_t)((g + 1) % SPEC_LISTS) * db.B;
    da.defer = db.defer + b; da.tag = tag;
    da.b = b; da.n = n; da.K = SPEC_K; da.iteration = iteration; da.round = round; da.q0 = q0; da.tile = db.tile;
    sAcc[0] = spec_decide(da, sRes);
  }
  __syncthreads();
  const int accepted = sAcc[0];
  if (accepted >= 0) { /* discardTop(): the accepted trial state becomes the band (same arithmetic as the tile tasks) */
    const double* adx = dx_of(accepted);
    const bool ok = sRes[accepted * RES_STRIDE + 5] != 0.0;
    for (int r = tid; r < N; r += nthreads) {
      if (!row_is_real(r, n)) continue;
      const double dxv = ok ? __ldcg(adx + (size_t)r * 32) : sB[r];
      const double xv = sP0[r] + dxv;
      gP[r] = ((r & 3) == 2) ? normalize_theta(xv) : xv;
    }
  }
}

}  // namespace tebgpu
