/*
 * teb_solve_warp.cuh — k_solve_warp: ONE WARP per (band, trial) system, for the latency regime (a single planning
 * request: a few hundred systems on 148 SMs, where a thread-per-system solver leaves the machine empty and each thread
 * crawls at its own fp64 issue rate: ~75 dependent-latency DFMA per pivot).
 *
 * Same factorisation as k_solve_tpb - right-looking banded LDL^T, half bandwidth 10, lu = c_u / d,
 * W[u][q] -= lu c_q, y_u -= lu y_j - so factors and solutions are bit-identical; only the mapping differs:
 *   * the live 11 x 11 window (lower triangle) and the 11 live right-hand-side entries are spread over the 32 lanes:
 *     lane (m, p), m = lane & 15, p = lane >> 4, owns the entries whose COLUMN index is congruent to m modulo 16 and
 *     whose diagonal offset k = row - column has parity p (register t <-> k = 2 t + p; k = 11 is the rhs, keyed by its
 *     row). Ownership never moves: an entry is born (loaded) and dies (eliminated) in the same lane and register.
 *   * per pivot the two lanes holding column j publish it (d, c_1 .. c_10, y_j) through a 12-double shared-memory
 *     buffer (double buffered: one __syncwarp per pivot); every lane then updates its <= 6 entries with two multiplies
 *     each. Rows of H enter through a cp.async ring 16 rows ahead.
 *   * the factor is written in ROW form (z_j, L[j][j-1 .. j-10]), which turns the back substitution into axpy steps:
 *     once x_R is known it is broadcast and every lane updates the one accumulator it owns (row r = lane mod 16 inside the
 *     window): a shuffle and one FMA per row on the dependent chain.
 * Writes dx / res in the layout k_trial_eval2 reads, so the rest of the LM iteration is unchanged.
 *
 * MEASURED (profiles/r2_history.md): 0.74 ms per solve of a 32-candidate request at 200 poses against 0.26 ms of
 * k_solve_tpb - the per-pivot chain here (publish -> __syncwarp -> shared-memory load -> fp64 divide -> update ->
 * cp.async wait -> __syncwarp) is longer than the register-resident chain of a single thread, and the fp64 divide sits
 * on both. The kernel is therefore NOT the default; it stays as a second, independently mapped implementation of the
 * factorisation whose results must be (and are) bit-identical.
 * Replaces LinearSolverCSparse::solve (optimal_planner.cpp:169-172) like k_solve_tpb.
 */
#pragma once

#include "teb_spec.cuh"

namespace tebgpu {

constexpr int SW_WARPS = 4;          /* systems per CTA */
constexpr int SW_RING = 32;          /* rows in the cp.async ring (H rows forward, factor rows backward) */
constexpr int SW_AHEAD = 16;         /* prefetch distance in rows */
constexpr int SW_SMEM_PER_WARP = SW_RING * HROW + 2 * 12 + 16 * 12; /* doubles */

__global__ void __launch_bounds__(32 * SW_WARPS) k_solve_warp(DevBatch db, SpecBufs sp, int iteration, int round, int g) {
  __shared__ __align__(16) double sw_mem[SW_WARPS * SW_SMEM_PER_WARP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int t = blockIdx.x * SW_WARPS + warp;        /* system index = K * slot + k, as in k_solve_tpb */
  const int SPEC_K = sp.K;
  const int slot = t / SPEC_K;
  const int k = t - slot * SPEC_K;
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return;                                  /* whole warp */
  const BandState* st = &db.state[b];
  if (!st->active) return;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  if (q0 + k >= 10) return;
  const int n = db.n[b];
  const int N = 4 * n;
  double lambda, ni;
  if (round == 0 && iteration == 0) { lambda = band_lambda_init(db, b, n); ni = 2; }
  else { lambda = st->lambda; ni = st->ni; }
  spec_lambda(lambda, ni, k);

  double* ring = sw_mem + (size_t)warp * SW_SMEM_PER_WARP;   /* [SW_RING][12] */
  double* col = ring + SW_RING * HROW;                       /* [2][12] pivot column: d, c_1..c_10, y_j */
  double* Lrow = col + 24;                                   /* [16][12] row-form factor rows under construction */
  const double* gH = db.Hb + (size_t)b * 4 * db.n_cap * HROW;
  double* gF = sp.Lf + (size_t)t * 4 * db.n_cap * HROW;      /* this system's factor rows [row][12] */
  double* gx = sp.dx + (size_t)(t >> 5) * 32 * 4 * db.n_cap + (t & 31); /* + r * 32: layout of k_trial_eval2 */
  double* res = sp.res + ((size_t)b * SPEC_K_MAX + k) * RES_STRIDE;

  const int m = lane & 15, p = lane >> 4;
  const uint32_t ring_u32 = smem_u32(ring);
  auto prefetch_row = [&](const double* base, int r) { /* lanes 0..5: one 16-byte piece of the 96-byte row r */
    if (lane < 6) cp_async16(ring_u32 + (uint32_t)(((r & (SW_RING - 1)) * HROW + 2 * lane) * 8), base + (size_t)r * HROW + 2 * lane);
  };
  for (int e = lane; e < 16 * 12; e += 32) Lrow[e] = 0.0;
  /* rows 0 .. SW_AHEAD + 10 of H: the initial window and the first prefetch distance */
  for (int r = 0; r <= SW_AHEAD + 10; ++r) {
    if (r < N) prefetch_row(gH, r);
    cp_async_commit();
  }
  cp_async_wait<SW_AHEAD>();   /* rows 0 .. 10 have landed */
  __syncwarp();
  auto hval = [&](int r, int kk) -> double { /* H[r][r - kk] (kk <= 10, + lambda on real diagonals) or b[r] (kk = 11); identity beyond N */
    if (r >= N) return kk == 0 ? 1.0 : 0.0;
    double v = ring[(r & (SW_RING - 1)) * HROW + kk];
    if (kk == 0 && row_is_real(r, n)) v += lambda;
    return v;
  };
  double R[6];
#pragma unroll
  for (int tt = 0; tt < 6; ++tt) {
    const int kk = 2 * tt + p;
    R[tt] = 0.0;
    if (m <= 10) {
      if (kk <= 10) { if (m + kk <= 10) R[tt] = hval(m + kk, kk); }   /* entry (row m + kk, column m) */
      else R[tt] = hval(m, 11);                                       /* y_m */
    }
  }
  bool ok = true;
  int cur = 0;
  for (int j = 0; j < N; ++j) {
    const int s = j & 15;
    double* cb = col + 12 * cur;
    if (m == s) {
#pragma unroll
      for (int tt = 0; tt < 6; ++tt) cb[2 * tt + p] = R[tt];
    }
    __syncwarp();
    const double d = cb[0];
    if (!pivot_ok(d)) ok = false;
    const double inv = 1.0 / d;
    const double yj = cb[11];
    const int uC = (m - s) & 15;
    if (uC >= 1 && uC <= 10) {
      const double cq = cb[uC];
#pragma unroll
      for (int tt = 0; tt < 6; ++tt) {
        const int kk = 2 * tt + p;
        if (kk <= 10) {
          const int uR = uC + kk;
          if (uR <= 10) R[tt] -= (cb[uR] * inv) * cq;
        } else {
          R[tt] -= (cq * inv) * yj;          /* rhs of row j + uC */
        }
      }
    }
    /* factor: column j of L goes into the row records under construction; row j's own record is complete */
    if (lane >= 1 && lane <= 10) Lrow[((j + lane) & 15) * 12 + lane] = cb[lane] * inv;
    if (lane <= 11) {
      double v;
      if (lane == 0) v = yj * inv;                           /* z_j */
      else if (lane <= 10) v = Lrow[(j & 15) * 12 + lane];   /* L[j][j - lane], written at pivot j - lane */
      else v = inv;
      gF[(size_t)j * HROW + lane] = v;
    }
    /* row j + 11 enters the window (its ring slot was filled SW_AHEAD rows ago) */
    cp_async_wait<SW_AHEAD - 1>();
    __syncwarp();
    {
      const int rn = j + 11;
      const int k0 = (11 - uC) & 15;                         /* offset of the entering row in this lane's column */
      if (k0 <= 10 && (k0 & 1) == p) {
        const double v = hval(rn, k0);
        const int tsel = k0 >> 1;
#pragma unroll
        for (int tt = 0; tt < 6; ++tt)
          if (tt == tsel) R[tt] = v;
      }
      if (p == 1 && m == (rn & 15)) R[5] = hval(rn, 11);
    }
    {
      const int rp = j + 11 + SW_AHEAD;
      if (rp < N) prefetch_row(gH, rp);
      cp_async_commit();
    }
    cur ^= 1;
  }
  cp_async_wait<0>();
  if (lane == 0) { res[5] = ok ? 1.0 : 0.0; res[6] = lambda; }
  if (!ok) return; /* CSparse failure: k_trial_eval2 uses dx = b */
  __syncwarp();
  __threadfence_block();

  /* back substitution, axpy form: x_R = acc_R, then acc_{R-u} -= L[R][R-u] x_R for u = 1 .. 10. Lane l < 16 owns the
   * accumulator of the row r with r mod 16 = l that lies inside the window [R - 10, R]; it is created (= z_r) the first
   * time the row enters the window, i.e. at R = min(N - 1, r + 10), and receives its updates in the order u = 10 .. 1 -
   * the order of k_solve_tpb's dot product, so the solutions are bit-identical. */
  for (int c = 0; c <= SW_AHEAD; ++c) {
    const int r = N - 1 - c;
    if (r >= 0) prefetch_row(gF, r);
    cp_async_commit();
  }
  double acc = 0.0;
  for (int Rr = N - 1; Rr >= 0; --Rr) {
    cp_async_wait<SW_AHEAD - 10>();                          /* factor rows Rr .. Rr - 10 have landed */
    __syncwarp();
    const double* fr = ring + (Rr & (SW_RING - 1)) * HROW;
    const int u = (Rr - lane) & 15;                          /* this lane's row is Rr - u */
    const int r = Rr - u;
    const bool mine = lane < 16 && u <= 10 && r >= 0;
    if (mine && (u == 10 || Rr == N - 1)) acc = ring[(r & (SW_RING - 1)) * HROW]; /* z_r */
    const double xR = __shfl_sync(0xffffffffu, acc, Rr & 15);
    if (lane == (Rr & 15)) gx[(size_t)Rr * 32] = xR;
    if (mine && u >= 1) acc -= fr[u] * xR;
    const int rp = Rr - 1 - SW_AHEAD;
    if (rp >= 0) prefetch_row(gF, rp);
    cp_async_commit();
  }
  cp_async_wait<0>();
}

}  // namespace tebgpu
