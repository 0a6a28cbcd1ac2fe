/*
 * teb_solve_lat.cuh — k_solve_lat: the solver of the LATENCY regime (one planning request: a few hundred (band, trial)
 * systems). One warp per system, the whole system resident in shared memory, and a TWISTED factorisation: the top
 * half-warp eliminates the unknowns 0 .. m-1 downwards while the bottom half-warp eliminates N-1 .. m+11 upwards; the 11
 * unknowns in between (one full window, so the two sweeps never touch each other's pivots) are eliminated last by the
 * top half after the two Schur contributions have been added. This is the Cholesky (LDL^T) factorisation of P H P^T
 * for that elimination order - H is symmetric positive definite, so any order is stable without pivoting - and it
 * halves the dependent chain: ~N/2 + 11 pivots instead of N. The back substitution runs from the middle outwards, again
 * with both half-warps in lockstep.
 *
 * Why it exists: k_solve_tpb (one THREAD per system) needs 0.26 ms per solve of a 32-candidate, 200-pose request no
 * matter how few systems there are (800 pivots x ~75 DFMA issued by one thread), 85 % of that request's 6.3 ms. Here
 * the per-pivot work is spread over the lanes and the per-pivot chain is
 *     last update of the pivot (DFMA) -> shuffle of d -> reciprocal (MUFU + 2 Newton steps) -> l = c * inv -> DFMA
 * with the pivot column travelling through shared memory beside it.
 *
 * Mapping (per half-warp h, "sweep coordinates" q: unknown q for the top half, unknown N-1-q for the bottom half):
 *   * lane mm = lane & 15 owns the window column q with q mod 16 == mm: registers R[k] = entry (q + k, q), k = 0 .. 10,
 *     and Ry = right-hand side of q. Ownership never moves; the column that enters the window (q = t + 11) is gathered
 *     from the shared-memory copy of H by the lane whose registers have just become free.
 *   * per pivot t the owner publishes (d, c_1 .. c_10, y) in a double-buffered 12-double record; the lane that owns
 *     column t + u (u = 1 .. 10) subtracts c_{u+k} * l_u from its entries and y_t * l_u from its right-hand side.
 *   * the factor column (z_t = y_t / d, l_1 .. l_10) overwrites row `unknown(t)` of the shared-memory H (dead by then),
 *     so the factor never leaves the SM; only dx goes to global memory, in the layout k_trial_eval2 reads.
 *   * back substitution in axpy form: the lane that owns row r keeps acc_r = z_r - sum l_{r,u} x_{r+u}; once x_R is known
 *     it is broadcast by one shuffle and every live row takes one DFMA.
 * tools/twisted_model.py executes exactly this index arithmetic lane by lane on the CPU against a dense solve.
 *
 * The elimination order differs from k_solve_tpb's, so the solutions agree to rounding, not bit for bit; the LM
 * decisions and trajectories stay within the tolerances of tests/test_gpu_*.py. tests/test_gpu_solve.py checks every
 * mapping system by system against a long-double banded LDL^T: backward error <= 64 u, forward error <= 1e-13 relative
 * on well-conditioned systems and <= 64 u kappa on the others (kernel A's systems at lambda_0 reach kappa ~1e8).
 * Measured on a B200 (1000 W): < 5 u backward and <= 0.05 u kappa forward, alike for this kernel and k_solve_tpb.
 * Replaces LinearSolverCSparse::solve (optimal_planner.cpp:169-172), like k_solve_tpb.
 */
#pragma once

#include <math_constants.h>

#include "teb_spec.cuh"

namespace tebgpu {

constexpr int LAT_WAVES = 3;          /* automatic mode: k_solve_lat replaces k_solve_tpb while a round fits this many waves of
                                         resident CTAs (a wave takes ~1/4 of the time k_solve_tpb needs for any number of systems) */
constexpr int SL_REC = 24;            /* published pivot column: d, c_1 .. c_10 at [0..10], zeros at [11..21], y at [22] */
constexpr int SL_CB = 2 * 2 * SL_REC; /* [half][buffer] */
constexpr int SL_SPECIAL = 2 * HROW + SL_REC; /* an all-zero column, an identity column, the dummy record of the non-owners */
constexpr int SL_MID = 11 * HROW;     /* the bottom sweep's contribution to the middle block */
__host__ __device__ constexpr size_t solve_lat_smem_bytes(int n_cap) {
  return ((size_t)4 * n_cap * HROW + SL_CB + SL_SPECIAL + SL_MID) * sizeof(double) + 16;
}

/* 1 / d to ~1 ulp: MUFU.RCP64H seed (2^-20) and two Newton steps; d is a positive, normal pivot. One volatile block:
 * a lone warp issues in order, so WHERE the dependent chain sits in the instruction stream matters - it has to come
 * after the independent loads of the step, and the compiler must not move it. */
__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm volatile(
      "{ .reg .f64 e, y, nd;\n"
      "neg.f64 nd, %1;\n"
      "rcp.approx.ftz.f64 y, %1;\n"
      "fma.rn.f64 e, nd, y, 0d3FF0000000000000;\n"
      "fma.rn.f64 y, y, e, y;\n"
      "fma.rn.f64 e, nd, y, 0d3FF0000000000000;\n"
      "fma.rn.f64 %0, y, e, y; }"
      : "=d"(x)
      : "d"(d));
  return x;
}

/* predicated shared-memory accesses as single instructions: `if (p) { several stores }` becomes a divergent branch, and a
 * predicated load into a live register cannot be written in C++ at all */
__device__ __forceinline__ void st_shared_pred(uint32_t addr, double v, bool p) {
  asm volatile("{ .reg .pred q; setp.ne.b32 q, %2, 0; @q st.shared.f64 [%0], %1; }" ::"r"(addr), "d"(v), "r"((int)p) : "memory");
}
/* the 12 doubles of one record (column k = 0 .. 10, y) -> c[0..10], y, only in the lanes where p holds */
__device__ __forceinline__ void ld_column_pred(uint32_t addr, double (&c)[11], double& y, bool p) {
  asm volatile(
      "{ .reg .pred q; setp.ne.b32 q, %13, 0;\n"
      "@q ld.shared.v2.f64 {%0, %1}, [%12];\n"
      "@q ld.shared.v2.f64 {%2, %3}, [%12+16];\n"
      "@q ld.shared.v2.f64 {%4, %5}, [%12+32];\n"
      "@q ld.shared.v2.f64 {%6, %7}, [%12+48];\n"
      "@q ld.shared.v2.f64 {%8, %9}, [%12+64];\n"
      "@q ld.shared.v2.f64 {%10, %11}, [%12+80]; }"
      : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3]), "+d"(c[4]), "+d"(c[5]), "+d"(c[6]), "+d"(c[7]), "+d"(c[8]), "+d"(c[9]),
        "+d"(c[10]), "+d"(y)
      : "r"(addr), "r"((int)p)
      : "memory");
}
/* publish a pivot column: d, c_1 .. c_10 (and a zero) at [0..11], y at [22]. UNCONDITIONAL: the lanes that are not the
 * owner pass the address of a dummy record (same-address stores cost one wavefront). Seven predicated stores in a row get
 * turned into a divergent branch by ptxas, which puts a reconvergence barrier and a WARPSYNC on the pivot chain. */
__device__ __forceinline__ void st_record(uint32_t addr, const double (&c)[11], double y) {
  asm volatile(
      "{ .reg .f64 z; mov.f64 z, 0d0000000000000000;\n"
      "st.shared.v2.f64 [%12], {%0, %1};\n"
      "st.shared.v2.f64 [%12+16], {%2, %3};\n"
      "st.shared.v2.f64 [%12+32], {%4, %5};\n"
      "st.shared.v2.f64 [%12+48], {%6, %7};\n"
      "st.shared.v2.f64 [%12+64], {%8, %9};\n"
      "st.shared.v2.f64 [%12+80], {%10, z};\n"
      "st.shared.f64 [%12+176], %11; }" ::"d"(c[0]),
      "d"(c[1]), "d"(c[2]), "d"(c[3]), "d"(c[4]), "d"(c[5]), "d"(c[6]), "d"(c[7]), "d"(c[8]), "d"(c[9]), "d"(c[10]), "d"(y),
      "r"(addr)
      : "memory");
}
__device__ __forceinline__ void st_record_pred(uint32_t addr, const double (&c)[11], double y, bool p) {
  asm volatile(
      "{ .reg .pred q; .reg .f64 z; setp.ne.b32 q, %13, 0; mov.f64 z, 0d0000000000000000;\n"
      "@q st.shared.v2.f64 [%12], {%0, %1};\n"
      "@q st.shared.v2.f64 [%12+16], {%2, %3};\n"
      "@q st.shared.v2.f64 [%12+32], {%4, %5};\n"
      "@q st.shared.v2.f64 [%12+48], {%6, %7};\n"
      "@q st.shared.v2.f64 [%12+64], {%8, %9};\n"
      "@q st.shared.v2.f64 [%12+80], {%10, z};\n"
      "@q st.shared.f64 [%12+176], %11; }" ::"d"(c[0]),
      "d"(c[1]), "d"(c[2]), "d"(c[3]), "d"(c[4]), "d"(c[5]), "d"(c[6]), "d"(c[7]), "d"(c[8]), "d"(c[9]), "d"(c[10]), "d"(y),
      "r"(addr), "r"((int)p)
      : "memory");
}
/* ten consecutive elements of a published column and its y: one block, so that the loads are issued back to back and
 * land together instead of one by one in front of the multiply that needs them */
__device__ __forceinline__ void ld_record(uint32_t addr, uint32_t yaddr, double (&c)[10], double& y) {
  asm volatile(
      "ld.shared.f64 %0, [%11];\n"
      "ld.shared.f64 %1, [%11+8];\n"
      "ld.shared.f64 %2, [%11+16];\n"
      "ld.shared.f64 %3, [%11+24];\n"
      "ld.shared.f64 %4, [%11+32];\n"
      "ld.shared.f64 %5, [%11+40];\n"
      "ld.shared.f64 %6, [%11+48];\n"
      "ld.shared.f64 %7, [%11+56];\n"
      "ld.shared.f64 %8, [%11+64];\n"
      "ld.shared.f64 %9, [%11+72];\n"
      "ld.shared.f64 %10, [%12];"
      : "=d"(c[0]), "=d"(c[1]), "=d"(c[2]), "=d"(c[3]), "=d"(c[4]), "=d"(c[5]), "=d"(c[6]), "=d"(c[7]), "=d"(c[8]), "=d"(c[9]), "=d"(y)
      : "r"(addr), "r"(yaddr)
      : "memory");
}

/* TEBGPU_LAT_TIMING=1: block 0 prints the cycles of its phases (device printf; diagnostics only) */
__device__ int g_lat_timing = 0;

__global__ void __launch_bounds__(32, 1) k_solve_lat(DevBatch db, SpecBufs sp, int iteration, int round, int g) {
  extern __shared__ __align__(128) unsigned char sl_raw[];
  const int lane = threadIdx.x;
  const int t_sys = blockIdx.x;                       /* system index = K * slot + k, as in k_solve_tpb */
  const int SPEC_K = sp.K;
  const int slot = t_sys / SPEC_K;
  const int k_trial = t_sys - slot * SPEC_K;
  if (round > 0 && sp.lat_cap > 0 && !retry_round_takes_lat(sp, round, g)) return; /* list too long: k_solve_tpb does this round */
  const int b = spec_band(db, sp, round, g, slot);
  if (b < 0) return;                                  /* whole warp */
  const BandState* st = &db.state[b];
  if (!st->active) return;
  const int q0 = (round == 0) ? 0 : sp.qmax[b];
  if (q0 + k_trial >= 10) return;
  const int n = db.n[b];
  const int N = 4 * n;
  double lambda, ni;
  if (round == 0 && iteration == 0) { lambda = band_lambda_init(db, b, n); ni = 2; }
  else { lambda = st->lambda; ni = st->ni; }
  spec_lambda(lambda, ni, k_trial);

  double* Hs = reinterpret_cast<double*>(sl_raw);                 /* [N][12]: columns of H, overwritten by the factor */
  double* cball = Hs + (size_t)4 * db.n_cap * HROW;
  double* special = cball + SL_CB;
  double* mid = special + SL_SPECIAL;
  uint64_t* bar = reinterpret_cast<uint64_t*>(mid + SL_MID);
  const double* gH = db.Hb + (size_t)b * 4 * db.n_cap * HROW;
  double* gx = sp.dx + (size_t)(t_sys >> 5) * 32 * 4 * db.n_cap + (t_sys & 31); /* + r * 32: layout of k_trial_eval2 */
  double* res = sp.res + ((size_t)b * SPEC_K_MAX + k_trial) * RES_STRIDE;

  const long long c_start = clock64();
  if (lane == 0) { mbar_init(bar, 1); mbar_fence_init(); }
  __syncwarp();
  if (lane == 0) {
    const uint32_t bytes = (uint32_t)N * HROW * sizeof(double);
    mbar_expect_tx(bar, bytes);
    tma_load_1d(Hs, gH, bytes, bar);
  }
  const int h = lane >> 4, mm = lane & 15;
  const int m = (N - 11 + 1) / 2;            /* top sweep: pivots 0 .. m-1, then the middle m .. m+10 */
  const int T_bot = N - 11 - m;              /* bottom sweep: pivots N-1 .. m+11 (T_bot <= m) */
  const int src_base = lane & 16;
  for (int e = lane; e < SL_CB + SL_SPECIAL; e += 32) cball[e] = (e == SL_CB + HROW) ? 1.0 : 0.0;
  mbar_wait(bar, 0);
  const long long c_loaded = clock64();

  /* One pass over the resident copy turns it into what the sweeps read with six 16-byte loads per column:
   *   rows 0 .. m+10 (top sweep + middle): row q becomes COLUMN q of the leading block, Hc[q][k] = H[q+k][q] (zero when
   *   q + k leaves the block); rows m+11 .. N-1 stay as they are - row c, H[c][c-k], IS column c of the mirrored
   *   problem, and c - k >= m always holds there. lambda is added to the real diagonals, the right-hand side stays at
   *   [11]. Done in chunks of 32 rows, ascending: a chunk reads rows of its own and the next chunk only. */
  {
    const int top_rows = m + 11;
    /* lane l reads element k = (j + l / 4) mod 11 of its column in step j: rows are 96 bytes apart, so with one k for
     * the whole warp eight lanes would hit every bank (8-way conflict, 16 wavefronts per access); staggering k by l / 4
     * spreads the 32 accesses over all banks (2 wavefronts, the minimum for 256 bytes) */
    const int kst = lane >> 2;
    for (int q0r = 0; q0r < top_rows; q0r += 32) {
      const int q = q0r + lane;
      double v[11];
      const bool is_top = q < top_rows;
      const bool real = is_top && row_is_real(q, n);
#pragma unroll
      for (int j = 0; j < 11; ++j) {
        int k = j + kst;
        k = k >= 11 ? k - 11 : k;
        const bool on = is_top && q + k < top_rows;
        const double x = Hs[on ? (q + k) * HROW + k : 0];
        v[j] = on ? x : 0.0;
        if (k == 0 && real) v[j] += lambda;
      }
      __syncwarp();
      if (is_top) {
#pragma unroll
        for (int j = 0; j < 11; ++j) {
          int k = j + kst;
          k = k >= 11 ? k - 11 : k;
          Hs[q * HROW + k] = v[j];
        }
      }
      __syncwarp();
    }
    for (int q = top_rows + lane; q < N; q += 32)
      if (row_is_real(q, n)) Hs[q * HROW] += lambda;
    __syncwarp();
  }

  /* the shared-window base goes through an opaque move: otherwise the compiler re-derives it inside the loops (an S2R of the
   * CTA-in-cluster id per use, a variable-latency instruction in front of every address) */
  uint32_t hs_u32 = smem_u32(Hs);
  asm volatile("mov.u32 %0, %0;" : "+r"(hs_u32));
  const uint32_t cb_u32 = hs_u32 + (uint32_t)(4 * db.n_cap * HROW + h * 2 * SL_REC) * 8u;
  const uint32_t zero_u32 = hs_u32 + (uint32_t)(4 * db.n_cap * HROW + SL_CB) * 8u, ident_u32 = zero_u32 + HROW * 8;
  const uint32_t dummy_u32 = ident_u32 + HROW * 8;
  /* address of column q (sweep coordinates) of this half: the unknown's row, or the identity / zero column once the
   * sweep has left its own block (top: q >= m + 11, bottom: unknown < m + 11) */
  auto col_addr = [&](int q) -> uint32_t {
    const int un = h ? N - 1 - q : q;
    const bool inside = h ? un >= m + 11 : un < m + 11;
    return inside ? hs_u32 + (uint32_t)un * (HROW * 8) : (h ? zero_u32 : ident_u32);
  };

  /* lane mm holds column mm; from then on the lane that was the pivot one step ago (uC == 15) loads column t + 15 */
  double R[11], Ry = 0.0;
#pragma unroll
  for (int k = 0; k < 11; ++k) R[k] = 0.0;
  ld_column_pred(col_addr(mm), R, Ry, true);
  /* failure detection (pivot_ok, teb_spec.cuh) costs two integer instructions per pivot here: the smallest and the largest
   * high word of the pivots, as signed integers. Every pivot is a positive normal number iff the smallest is at least
   * 0x00100000 (a sign bit makes it negative; zero and subnormals lie below) and the largest is below 0x7ff00000 (inf,
   * NaN). */
  int hi_min = 0x3ff00000, hi_max = 0x3ff00000;
  const long long c_prep = clock64();

  /* Order inside a step (a lone warp issues in order, so the stream is laid out by hand and pinned with volatile asm):
   * shuffle of the pivot -> publish -> record loads -> column fetch -> [reciprocal chain] -> updates -> factor store.
   * Everything independent of 1/d is in flight before the reciprocal chain starts. */
  auto step = [&](int t, bool act) {
    const int s = t & 15;
    const int uC = (mm - s) & 15;
    const uint32_t cbt = cb_u32 + (uint32_t)(t & 1) * (SL_REC * 8);
    const double d = __shfl_sync(0xffffffffu, R[0], s | src_base);
    st_record((act && uC == 0) ? cbt : dummy_u32, R, Ry);
    __syncwarp();
    const bool upd = act && uC >= 1 && uC <= 10;
    const int ui = upd ? uC : 0;
    double ck[10], yj;
    ld_record(cbt + (uint32_t)ui * 8u, cbt + 22 * 8, ck, yj);
    /* the lane whose column was eliminated in the previous step fetches its next one, 15 columns ahead */
    ld_column_pred(col_addr(t + 15), R, Ry, uC == 15);
    const int dhi = act ? __double2hiint(d) : 0x3ff00000;
    hi_min = min(hi_min, dhi);
    hi_max = max(hi_max, dhi);
    const double inv = fast_rcp(d);
    const double lq = upd ? ck[0] * inv : 0.0;   /* exact no-op for the lanes that do not take part (0 * inf would not be) */
#pragma unroll
    for (int k = 0; k < 10; ++k) R[k] -= ck[k] * lq;      /* entries beyond c_10 read the record's zeros */
    Ry -= yj * lq;
    /* factor column of pivot t: z_t, l_1 .. l_10 into the dead row of H */
    {
      const int row = h == 0 ? t : N - 1 - t;
      st_shared_pred(hs_u32 + (uint32_t)(row * HROW + (uC <= 10 ? uC : 0)) * 8u, (uC == 0) ? yj * inv : lq, act && uC <= 10);
    }
  };

  /* Main part, unrolled by the ownership period of 16 steps: while both sweeps are active and the fetched column
   * (t + 15) lies inside the sweep's own block, everything that depends on (t mod 16, lane) - roles, record offsets,
   * the source lane of the shuffle - is a per-lane constant of the unrolled body, and the addresses of the fetched column
   * and of the factor row advance by one row per step. That takes ~25 integer instructions per step off a lone,
   * in-order warp. The remaining steps (< 16 + 15 at the end of the sweeps, the middle block) use the generic step. */
  const int nblk = T_bot > 15 ? (T_bot - 15) / 16 : 0;
  const int rt_zero = (int)special[0];   /* a zero the assembler cannot see through */
  {
    const uint32_t rstep = h ? (uint32_t)(-(HROW * 8)) : (uint32_t)(HROW * 8);
    uint32_t colp = hs_u32 + (uint32_t)(h ? N - 1 - 15 : 15) * (HROW * 8);
    uint32_t facp = hs_u32 + (uint32_t)(h ? N - 1 : 0) * (HROW * 8);
    for (int blk = 0; blk < nblk; ++blk) {
#pragma unroll
      for (int S = 0; S < 16; ++S) {
        const int uC = (mm - S - rt_zero) & 15;
        const uint32_t cbt = cb_u32 + (uint32_t)(S & 1) * (SL_REC * 8);
        const double d = __shfl_sync(0xffffffffu, R[0], S | src_base);
        st_record_pred(cbt, R, Ry, uC == 0);
        __syncwarp();
        const bool upd = (unsigned)(uC - 1) < 10u;
        double ck[10], yj;
        ld_record(cbt + (uint32_t)(upd ? uC : 0) * 8u, cbt + 22 * 8, ck, yj);
        ld_column_pred(colp, R, Ry, uC == 15);
        colp += rstep;
        hi_min = min(hi_min, __double2hiint(d));
        hi_max = max(hi_max, __double2hiint(d));
        const double inv = fast_rcp(d);
        const double lq = upd ? ck[0] * inv : 0.0;
#pragma unroll
        for (int k = 0; k < 10; ++k) R[k] -= ck[k] * lq;
        Ry -= yj * lq;
        st_shared_pred(facp + (uint32_t)(uC <= 10 ? uC : 0) * 8u, (uC == 0) ? yj * inv : lq, uC <= 10);
        facp += rstep;
      }
    }
  }
  for (int t = nblk * 16; t < m; ++t) step(t, h == 0 || t < T_bot);

  /* merge: the bottom window now holds the bottom sweep's contribution to the middle block (its columns
   * q' = T_bot .. T_bot + 10 are the unknowns m + 10 .. m); add it to the top window */
  {
    if (h == 1) {
      const int i = (mm - T_bot) & 15;
      if (i <= 10) {
        const int a = 10 - i;                /* unknown m + a */
#pragma unroll
        for (int k = 0; k < 11; ++k)
          if (a - k >= 0) mid[a * HROW + k] = R[k];
        mid[a * HROW + 11] = Ry;
      }
    }
    __syncwarp();
    if (h == 0) {
      const int i = (mm - m) & 15;
      if (i <= 10) {
#pragma unroll
        for (int k = 0; k < 11; ++k)
          if (i + k <= 10) R[k] += mid[(i + k) * HROW + k];
        Ry += mid[i * HROW + 11];
      }
    }
    __syncwarp();
  }
  for (int t = m; t < m + 11; ++t) step(t, h == 0);

  const long long c_fact = clock64();
  __syncwarp();

  /* ---- back substitution from the middle outwards, dot-product form: x_j = z_j - sum_u l_{j,u} x_{j+u}.
   * No communication at all: every lane of a half-warp computes the same values (the factor rows are broadcast reads),
   * all 32 lanes solve the middle block, then the top half walks down to unknown 0 and the bottom half up to N-1. The
   * ten most recent solutions live in a register ring whose indices are static after unrolling by ten; the newest one
   * enters the sum last, so the dependent chain per row is ONE FMA and a row costs its eleven fp64 instructions
   * (~28 cycles) instead of shuffle + FMA + bookkeeping (~90 cycles in the axpy form this replaced). */
  {
    double W[10];
#pragma unroll
    for (int k = 0; k < 10; ++k) W[k] = 0.0;
    /* row = (z, l_1 .. l_10, pad), loaded one row ahead of its use; x_{j+u} = W[(P + u) % 10], the new solution goes to
     * W[P]. Four partial sums keep the fp64 pipe busy without dependent stalls; x_{j+1} enters last. */
    struct Row { double2 f0, f1, f2, f3, f4, f5; };
    auto row_load = [&](const double* rowp) -> Row {
      const double2* r2 = reinterpret_cast<const double2*>(rowp);
      Row r;
      r.f0 = r2[0]; r.f1 = r2[1]; r.f2 = r2[2]; r.f3 = r2[3]; r.f4 = r2[4]; r.f5 = r2[5];
      return r;
    };
    auto row_solve = [&](const Row& r, int P) -> double {
      double a = fma(-r.f5.x, W[(P + 10) % 10], r.f0.x);
      double b = -r.f4.y * W[(P + 9) % 10];
      double c = -r.f4.x * W[(P + 8) % 10];
      double d = -r.f3.y * W[(P + 7) % 10];
      a = fma(-r.f3.x, W[(P + 6) % 10], a);
      b = fma(-r.f2.y, W[(P + 5) % 10], b);
      c = fma(-r.f2.x, W[(P + 4) % 10], c);
      d = fma(-r.f1.y, W[(P + 3) % 10], d);
      a = fma(-r.f1.x, W[(P + 2) % 10], a);
      return fma(-r.f0.y, W[(P + 1) % 10], (a + b) + (c + d));
    };
    /* the middle block m + 10 .. m (rows of the top sweep's factor), ring positions 9, 8, .., 0, 9 */
    double xm10 = 0.0;
    Row cur = row_load(Hs + (size_t)(m + 10) * HROW);
#pragma unroll
    for (int i = 0; i < 11; ++i) {
      const int P = (19 - i) % 10;
      const int j = m + 10 - i;
      /* next: the following middle row, or (after the last one) the first row of this half's outward walk */
      const Row nxt = row_load(Hs + (size_t)(i < 10 ? j - 1 : (h ? (T_bot > 0 ? m + 11 : 0) : m - 1)) * HROW);
      const double x = row_solve(cur, P);
      if (i == 0) xm10 = x;
      W[P] = x;
      if (lane == 0) gx[(size_t)j * 32] = x;
      cur = nxt;
    }
    /* the ring now holds x_m (position 9), x_{m+1} .. x_{m+9} (positions 0 .. 8): what the top half needs next at
     * position 8. The bottom half continues in its own sweep order: its x_{q'+u} is the unknown m + 11 - u. */
    {
      double Wb[10];
      Wb[9] = xm10;
#pragma unroll
      for (int k = 0; k < 9; ++k) Wb[k] = W[8 - k];
#pragma unroll
      for (int k = 0; k < 10; ++k) W[k] = h ? Wb[k] : W[k];
    }
    const int cnt = h ? T_bot : m;
    const int rinc = h ? HROW : -HROW;
    const double* rp = Hs + (size_t)(h ? m + 11 : m - 1) * HROW + rinc;   /* the row AFTER the one held in `cur` */
    int un = h ? m + 11 : m - 1;
    const int uinc = h ? 1 : -1;
    for (int i0 = 0; i0 < m; i0 += 10) {
#pragma unroll
      for (int ii = 0; ii < 10; ++ii) {
        const int P = (18 - ii) % 10;                     /* 8, 7, .., 0, 9 */
        const bool valid = i0 + ii < cnt;                 /* past the end of a sweep: harmless row, nothing stored */
        const Row nxt = row_load(i0 + ii + 1 < cnt ? rp : Hs);
        const double x = row_solve(cur, P);
        W[P] = x;
        if (valid && mm == 0) gx[(size_t)un * 32] = x;
        rp += rinc;
        un += uinc;
        cur = nxt;
      }
    }
  }
  {
    /* the solve succeeded iff every pivot was a positive normal number (pivot_ok); otherwise k_trial_eval2 uses dx = b,
     * as CSparse leaves it */
    const bool ok = __all_sync(0xffffffffu, hi_min >= 0x00100000 && hi_max < 0x7ff00000);
    if (lane == 0) { res[5] = ok ? 1.0 : 0.0; res[6] = lambda; }
  }
  if (g_lat_timing && blockIdx.x == 0 && lane == 0)
    printf("k_solve_lat N=%d cycles: load %lld, prepare %lld, factorise %lld (%.1f per pivot step), back-substitute %lld (%.1f per step)\n", N,
           c_loaded - c_start, c_prep - c_loaded, c_fact - c_prep, (double)(c_fact - c_prep) / (m + 11), clock64() - c_fact,
           (double)(clock64() - c_fact) / (m + 11));
}

}  // namespace tebgpu
