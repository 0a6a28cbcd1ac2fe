"""The LM linear solve of the default solver, system by system, against an extended-precision banded LDL^T.

Every LM trial solves (H + lambda_k I_real) dx = b, I_real the identity on the real unknowns (rows 0 .. 2 and
4n-4 .. 4n-1 are identity rows: the fixed start / goal poses and dt of the last pose). Three kernels do it:
k_solve_tpb (thread per system, mode 0), k_solve_warp (warp per system, mode 1, bit-identical to mode 0 by design) and
k_solve_lat (twisted factorisation, mode 3, the default of a single planning request). End to end the LM loop hides a
wrong or inaccurate dx - the trial is rejected and lambda escalates - so tebgpu_solve_system runs the solve alone, with
the optimizer's grid and kernel choice, and every system is checked here against `ldlt_banded`, a banded LDL^T in numpy
long double (64-bit mantissa).

The reference and its own tests run without a GPU; the comparisons are marked `gpu`.
"""
import fractions

import numpy as np
import pytest
import scipy.linalg

LD = np.longdouble
U = 2.0 ** -53      # unit roundoff of fp64
BW = 10             # half bandwidth
MODES = (0, 1, 3)   # k_solve_tpb, k_solve_warp, k_solve_lat


# ------------------------------------------------------------------ reference (CPU)
def row_is_real(n_rows, n):
    """mask [n_rows] of the real unknowns of a band with n poses (teb_kernels.cuh row_is_real); rows >= 4n: False"""
    r = np.arange(n_rows)
    i, c = r >> 2, r & 3
    return np.where(c == 3, i <= n - 2, (i >= 1) & (i <= n - 2))


def host_lambdas(lam0, ni0, K):
    """lambda_k of trial k = 0 .. K-1 after k rejections (spec_lambda: lambda *= ni, ni *= 2), fp64 as on the device"""
    lam0 = np.asarray(lam0, dtype=np.float64)
    out = np.empty(lam0.shape + (K,))
    lam, ni = lam0.copy(), np.broadcast_to(np.asarray(ni0, dtype=np.float64), lam0.shape).copy()
    for k in range(K):
        out[..., k] = lam
        lam = lam * ni
        ni = ni * 2
    return out


def band_matrix(Hb, n, lam):
    """-> (W [S][N][11], rhs [S][N]) long double: W[s][r][k] = A[r][r-k] of A = H + lam I_real. Rows from 4 n[s] on
    become decoupled identity rows (b = 0), so that systems of different n share one N; the padding of Hb there is
    never read (it may hold NaN)."""
    Hb = np.asarray(Hb)
    S, N = Hb.shape[0], Hb.shape[1]
    n = np.broadcast_to(np.asarray(n), (S,))
    W = np.zeros((S, N, BW + 1), dtype=LD)
    rhs = np.zeros((S, N), dtype=LD)
    for s in range(S):
        Ns = 4 * int(n[s])
        W[s, :Ns] = Hb[s, :Ns, :BW + 1].astype(LD)
        rhs[s, :Ns] = Hb[s, :Ns, 11].astype(LD)
        W[s, :Ns, 0] += np.where(row_is_real(Ns, int(n[s])), LD(lam[s]), LD(0))
        W[s, Ns:, 0] = 1
    for k in range(1, BW + 1):   # entries left of column 0 do not exist
        W[:, :k, k] = 0
    return W, rhs


def _factor(W):
    """banded LDL^T without pivoting: -> (L [S][N][11] with L[j][u] = l_{j+u, j}, D [S][N])"""
    A = W.copy()
    S, N = A.shape[:2]
    L = np.zeros_like(A)
    D = np.zeros((S, N), dtype=LD)
    with np.errstate(all="ignore"):
        for j in range(N):
            d = A[:, j, 0].copy()
            D[:, j] = d
            top = min(BW, N - 1 - j)
            if top == 0:
                continue
            # c_u = A[j+u][j], u = 1 .. top
            c = np.zeros((S, BW + 1), dtype=LD)
            for u in range(1, top + 1):
                c[:, u] = A[:, j + u, u]
            lu = c / d[:, None]
            L[:, j, 1:top + 1] = lu[:, 1:top + 1]
            for u in range(1, top + 1):
                # A[j+u][j+q] -= l_u c_q, q = 1 .. u: stored at A[j+u][u-q]
                A[:, j + u, 0:u] -= lu[:, u:u + 1] * c[:, u:0:-1]
    return L, D


def _solve_factored(L, D, rhs):
    S, N = D.shape
    y = rhs.astype(LD).copy()
    with np.errstate(all="ignore"):
        for j in range(N):
            top = min(BW, N - 1 - j)
            if top:
                y[:, j + 1:j + 1 + top] -= L[:, j, 1:top + 1] * y[:, j:j + 1]
        z = y / D
        x = np.zeros_like(z)
        for j in range(N - 1, -1, -1):
            top = min(BW, N - 1 - j)
            x[:, j] = z[:, j] - (L[:, j, 1:top + 1] * x[:, j + 1:j + 1 + top]).sum(axis=1) if top else z[:, j]
    return x


def band_matvec(W, x):
    """A x for the symmetric band matrix W (long double)"""
    S, N = W.shape[:2]
    x = np.asarray(x, dtype=LD)
    y = W[:, :, 0] * x
    for k in range(1, BW + 1):
        y[:, k:] += W[:, k:, k] * x[:, :-k]      # lower: A[r][r-k] x[r-k]
        y[:, :-k] += W[:, k:, k] * x[:, k:]      # upper: A[r-k][r] x[r]
    return y


def band_norm_inf(W):
    a = np.abs(W[:, :, 0]).copy()
    for k in range(1, BW + 1):
        a[:, k:] += np.abs(W[:, k:, k])
        a[:, :-k] += np.abs(W[:, k:, k])
    return a.max(axis=1)


def _inv_norm1_estimate(L, D, iters=5):
    """Hager / Higham 1-norm estimate of A^-1 (A symmetric: the 1- and inf-norms agree); a lower bound, in practice
    within a small factor and usually exact"""
    S, N = D.shape
    x = np.full((S, N), LD(1) / N)
    est = np.zeros(S, dtype=LD)
    done = np.zeros(S, dtype=bool)
    for _ in range(iters):
        y = _solve_factored(L, D, x)
        est = np.where(done, est, np.abs(y).sum(axis=1))
        xi = np.where(y >= 0, LD(1), LD(-1))
        z = _solve_factored(L, D, xi)
        zmax = np.abs(z).max(axis=1)
        done |= zmax <= (z * x).sum(axis=1)
        if done.all():
            break
        j = np.abs(z).argmax(axis=1)
        x = np.zeros((S, N), dtype=LD)
        x[np.arange(S), j] = 1
    return est


def ldlt_banded(Hb, n, lam, cond=True):
    """Solve (H + lam I_real) x = b for every system s of Hb [S][4 n_cap][12] (tebgpu_build_system's layout), n [S]
    (or one n), lam [S]: banded LDL^T without pivoting, half bandwidth 10, in long double.
    -> dict x [S][4 n_cap] (long double; rows >= 4 n are 0), min_pivot [S], all_pivots_positive [S], max_diag [S] (largest
    real diagonal of A), cond [S] (inf-norm condition estimate, NaN unless every pivot is positive)."""
    W, rhs = band_matrix(Hb, n, np.broadcast_to(np.asarray(lam, dtype=np.float64), (len(Hb),)))
    L, D = _factor(W)
    x = _solve_factored(L, D, rhs)
    S, N = D.shape
    nn = np.broadcast_to(np.asarray(n), (S,))
    real = np.stack([row_is_real(N, int(v)) for v in nn])
    pos = np.all(D > 0, axis=1)
    out = dict(x=x, min_pivot=D.min(axis=1), all_pivots_positive=pos, W=W, rhs=rhs,
               max_diag=np.where(real, np.abs(W[:, :, 0]), LD(0)).max(axis=1))
    if cond:
        with np.errstate(all="ignore"):
            kappa = band_norm_inf(W) * _inv_norm1_estimate(L, D)
        out["cond"] = np.where(pos, kappa, np.nan)
    return out


def pack_dense(Hd, bd, n):
    """dense normal equations of the 4n-7 real unknowns -> one band [4n][12] with the identity rows
    (tests/test_gpu_parity.py _padded_from_dense)"""
    Nr = 4 * n - 7
    Hb = np.zeros((4 * n, 12))
    Hb[:, 0] = 1.0
    for r in range(Nr):
        for k in range(min(r, BW) + 1):
            Hb[r + 3, k] = Hd[r, r - k]
        Hb[r + 3, 11] = bd[r]
    return Hb


# ------------------------------------------------------------------ system generators
def _jjt_band(J):
    """A = J J^T for J [S][Nr][P] lower banded (J[r][p] = J[r][r-p], P <= 11): half bandwidth P - 1. -> [S][Nr][11]"""
    S, Nr, P = J.shape
    A = np.zeros((S, Nr, BW + 1))
    for k in range(min(BW, Nr - 1) + 1):
        for p in range(k, min(k + P, BW + 1)):
            # A[r][r-k] += J[r][r-p] J[r-k][r-p]; q = p - k is the offset of column r-p in row r-k
            q = p - k
            if q >= P or p >= P:
                continue
            A[:, k:, k] += J[:, k:, p] * J[:, :Nr - k, q]
    for k in range(1, BW + 1):
        A[:, :k, k] = 0
    return A


def embed(A_real, b_real, n, n_cap, pad=np.nan):
    """real block [S][4n-7][11] + rhs -> Hb [S][4 n_cap][12]: identity rows 0..2 and 4n-4..4n-1, rows 4n.. = pad"""
    S, Nr = A_real.shape[:2]
    assert Nr == 4 * n - 7
    Hb = np.zeros((S, 4 * n_cap, 12))
    Hb[:, :4 * n, 0] = 1.0
    Hb[:, 3:3 + Nr, :BW + 1] = A_real
    Hb[:, 3:3 + Nr, 11] = b_real
    Hb[:, 4 * n:, :] = pad
    return Hb


def spd_real_block(rng, S, n, ridge=0.1, rank_drop=0):
    """random J J^T + ridge * mean diag on the 4n-7 real unknowns, J lower banded with half bandwidth 10 so that every
    diagonal of the band is populated; rank_drop > 0 zeroes every rank_drop-th column of J first (a rank-deficient
    J J^T)"""
    Nr = 4 * n - 7
    J = rng.uniform(-1, 1, (S, Nr, BW + 1))
    for p in range(1, BW + 1):
        J[:, :p, p] = 0
    if rank_drop:
        for c in range(0, Nr, rank_drop):   # column c of J: entries J[c+p][p]
            for p in range(BW + 1):
                if c + p < Nr:
                    J[:, c + p, p] = 0
    A = _jjt_band(J)
    A[:, :, 0] += ridge * A[:, :, 0].mean(axis=1, keepdims=True)
    b = rng.uniform(-1, 1, (S, Nr))
    return A, b


def graded(A, b, rng, span=6.0):
    """D A D, D b with D = 10^uniform(-span, span) per unknown"""
    S, Nr = A.shape[:2]
    dexp = rng.uniform(-span, span, (S, Nr))
    D = 10.0 ** dexp
    A2 = A.copy()
    for k in range(BW + 1):
        A2[:, k:, k] *= D[:, k:] * D[:, :Nr - k]
    return A2, b * D


def dense_from_band(Wr):
    Nr = Wr.shape[0]
    A = np.zeros((Nr, Nr), dtype=Wr.dtype)
    for r in range(Nr):
        for k in range(min(r, BW) + 1):
            A[r, r - k] = A[r - k, r] = Wr[r, k]
    return A


# ------------------------------------------------------------------ CPU tests of the reference
def _exact_solve(A, b, shift):
    """Gaussian elimination in exact rationals on A + diag(shift)"""
    N = len(b)
    M = [[fractions.Fraction(float(A[i, j])) for j in range(N)] + [fractions.Fraction(float(b[i]))] for i in range(N)]
    for i in range(N):
        M[i][i] += fractions.Fraction(float(shift[i]))
    for c in range(N):
        p = next(r for r in range(c, N) if M[r][c] != 0)
        M[c], M[p] = M[p], M[c]
        for r in range(c + 1, N):
            f = M[r][c] / M[c][c]
            if f:
                for k in range(c, N + 1):
                    M[r][k] -= f * M[c][k]
    x = [fractions.Fraction(0)] * N
    for r in range(N - 1, -1, -1):
        x[r] = (M[r][N] - sum(M[r][k] * x[k] for k in range(r + 1, N))) / M[r][r]
    return x


@pytest.mark.parametrize("n", range(3, 9))
def test_reference_matches_exact_rational_solve(n):
    """small systems, lambda on the real diagonal: long double result within 1e-17 of the exact solution (fp64 could not)"""
    rng = np.random.default_rng(100 + n)
    A, b = spd_real_block(rng, 2, n, ridge=0.05)
    Hb = embed(A, b, n, n)
    lam = np.array([0.0, 0.37])
    ref = ldlt_banded(Hb, n, lam)
    for s in range(2):
        Afull = np.eye(4 * n)
        Afull[3:4 * n - 4, 3:4 * n - 4] = dense_from_band(A[s])
        shift = np.where(row_is_real(4 * n, n), lam[s], 0.0)
        bfull = np.zeros(4 * n)
        bfull[3:4 * n - 4] = b[s]
        xe = np.array([LD(float(v)) + LD(float(v - fractions.Fraction(float(v)))) for v in _exact_solve(Afull, bfull, shift)])
        err = np.abs(ref["x"][s] - xe).max() / np.abs(xe).max()
        assert err <= 1e-17, (n, s, err)
        assert ref["all_pivots_positive"][s]
        # the condition estimate against the exact inf-norm condition number (Hager's estimate is a lower bound)
        Afull += np.diag(shift)
        kex = np.abs(Afull).sum(axis=1).max() * np.abs(np.linalg.inv(Afull)).sum(axis=1).max()
        assert kex / 10 <= float(ref["cond"][s]) <= kex * (1 + 1e-9), (kex, ref["cond"][s])


@pytest.mark.parametrize("n", [20, 57, 128])
def test_reference_matches_scipy_solveh_banded(n):
    rng = np.random.default_rng(n)
    A, b = spd_real_block(rng, 3, n, ridge=0.02)
    lam = np.array([1e-3, 0.5, 7.0])
    Hb = embed(A, b, n, n + 5)
    ref = ldlt_banded(Hb, n, lam)
    Nr = 4 * n - 7
    for s in range(3):
        ab = np.zeros((BW + 1, Nr))
        for k in range(BW + 1):
            ab[k, :Nr - k] = A[s, k:, k]
        ab[0] += lam[s]
        xs = scipy.linalg.solveh_banded(ab, b[s], lower=True)
        x = ref["x"][s]
        assert np.all(x[:3] == 0) and np.all(x[4 * n - 4:] == 0)
        assert np.abs(x[3:3 + Nr].astype(np.float64) - xs).max() <= 1e-12 * np.abs(xs).max()


def test_reference_pack_dense_layout():
    """pack_dense (the layout kernel A writes) and embed agree, and the packed system solves the dense one"""
    rng = np.random.default_rng(7)
    n = 9
    A, b = spd_real_block(rng, 1, n)
    Hd = dense_from_band(A[0])
    Hb = pack_dense(Hd, b[0], n)
    assert np.array_equal(Hb, embed(A, b, n, n)[0])
    ref = ldlt_banded(Hb[None], n, [0.0])
    x = np.linalg.solve(Hd, b[0])
    assert np.abs(ref["x"][0, 3:4 * n - 4].astype(np.float64) - x).max() <= 1e-13 * np.abs(x).max()


def test_reference_inertia_of_shifted_systems():
    """A - sigma I_real: every pivot positive iff sigma is below the smallest eigenvalue (Sylvester's law of inertia)"""
    rng = np.random.default_rng(3)
    n = 30
    A, b = spd_real_block(rng, 1, n, ridge=0.05)
    Hb = embed(A, b, n, n)
    ab = np.zeros((BW + 1, 4 * n - 7))
    for k in range(BW + 1):
        ab[k, :4 * n - 7 - k] = A[0, k:, k]
    emin = scipy.linalg.eigvals_banded(ab, lower=True, select="i", select_range=(0, 0))[0]
    for f, want in ((0.9, True), (1.1, False), (3.0, False)):
        ref = ldlt_banded(Hb, n, [-f * emin], cond=False)
        assert bool(ref["all_pivots_positive"][0]) is want


def test_reference_power_of_two_scaling_is_exact():
    rng = np.random.default_rng(5)
    n = 12
    A, b = spd_real_block(rng, 1, n)
    Hb = embed(A, b, n, n)
    r0 = ldlt_banded(Hb, n, [0.25])
    for e in (-200, 200):
        Hs = Hb * 2.0 ** e
        Hs[:, :, 0] = np.where(row_is_real(4 * n, n), Hs[0, :, 0], 1.0)
        r = ldlt_banded(Hs, n, [0.25 * 2.0 ** e])
        assert np.array_equal(r["x"], r0["x"])


def test_host_lambdas_is_spec_lambda():
    assert host_lambdas(1.5, 2.0, 5).tolist() == [1.5, 3.0, 12.0, 96.0, 1536.0]


# ------------------------------------------------------------------ GPU comparisons
_REPORT = {}


def _report(mode, what, value):
    key = (mode, what)
    _REPORT[key] = max(_REPORT.get(key, 0.0), float(value))
    print(f"[solve mode {mode}] worst {what} so far: {_REPORT[key]:.3e}")


@pytest.fixture(scope="module")
def gpu():
    import teb_local_planner_b200 as T
    g = T.TebGpu(128, 512, 1, 1, 0)
    yield g
    print("\nworst errors per solve mapping (mode 0 k_solve_tpb, 1 k_solve_warp, 3 k_solve_lat):")
    for (mode, what), v in sorted(_REPORT.items()):
        print(f"  mode {mode}  {what:>16s}  {v:.3e}")
    g.close()


def _run_modes(g, Hb, n, lam0, ni0, K):
    out = {}
    for mode in MODES:
        g.set_warp_solver(mode)
        out[mode] = g.solve_system(Hb, n, lam0, ni0, K)
    g.set_warp_solver(4)
    return out


def _check(g, Hb, n, lam0, ni0, K, fwd=None, name=""):
    """Run all three mappings on the batch and assert the properties of the module docstring.
    fwd: None (no forward-error check), 'tight' (1e-13 relative), 'cond' (64 u kappa relative) or 'tight_or_cond'
    (the larger of the two).
    Returns (results by mode, reference, host lambdas [B][K])."""
    Hb = np.ascontiguousarray(Hb, dtype=np.float64)
    B, rows = Hb.shape[:2]
    n = np.broadcast_to(np.asarray(n, dtype=np.int32), (B,)).copy()
    lam0 = np.broadcast_to(np.asarray(lam0, dtype=np.float64), (B,)).copy()
    ni0 = np.broadcast_to(np.asarray(ni0, dtype=np.float64), (B,)).copy()
    assert (B * K) % 32 != 0 or name.startswith("aligned"), "batches are sized so that the trials of a band straddle warps"
    lam_k = host_lambdas(lam0, ni0, K)                                    # [B][K]
    res = _run_modes(g, Hb, n, lam0, ni0, K)
    # reference: one system per (band, trial)
    Hs = np.repeat(Hb, K, axis=0)
    ns = np.repeat(n, K)
    ref = ldlt_banded(Hs, ns, lam_k.reshape(-1), cond=fwd in ("cond", "tight_or_cond"))
    xr = ref["x"].reshape(B, K, rows)
    pos = ref["all_pivots_positive"].reshape(B, K)
    clear = ((ref["min_pivot"] > 1e-8 * ref["max_diag"]) | (ref["min_pivot"] <= 0)).reshape(B, K)
    W, rhs = ref["W"], ref["rhs"]
    real_mask = np.stack([row_is_real(rows, int(v)) for v in ns]).reshape(B, K, rows)
    inside = (np.arange(rows)[None, :] < 4 * n[:, None])[:, None, :]     # [B][1][rows]
    dx0, ok0, lu0 = res[0]
    for mode, (dx, ok, lam_used) in res.items():
        tag = f"{name} mode {mode}"
        # 4. damping sequence, bit for bit
        assert np.array_equal(lam_used.view(np.uint64), lam_k.view(np.uint64)), tag
        # 5. failure flag: the same in every mapping, and what the reference's pivots say wherever they are clear
        assert np.array_equal(ok, ok0), (tag, np.argwhere(ok != ok0)[:8])
        bad = clear & (ok.astype(bool) != pos)
        assert not bad.any(), (tag, np.argwhere(bad)[:8], ref["min_pivot"].reshape(B, K)[bad][:8])
        good = ok.astype(bool)
        # 7. the kernel writes rows 0 .. 4n-1 and nothing after them; no NaN of the padding reaches the solution
        assert np.all(np.isnan(dx[np.broadcast_to(~inside, dx.shape)])), tag
        sol = np.where(inside, dx, 0.0)
        assert np.all(np.isfinite(sol[good])), tag
        # 6. identity rows: exactly zero
        ident = inside & ~real_mask
        assert np.all(sol[good][ident[good]] == 0.0), tag
        if not good.any():
            continue
        # 1. backward error in long double
        dxl = sol.reshape(B * K, rows).astype(LD)
        r = band_matvec(W, dxl) - rhs
        den = band_norm_inf(W) * np.abs(dxl).max(axis=1) + np.abs(rhs).max(axis=1)
        berr = (np.abs(r).max(axis=1) / den).reshape(B, K)[good]
        _report(mode, "backward/u", berr.max() / U)
        assert berr.max() <= 64 * U, (tag, berr.max() / U)
        # 2. forward error
        if fwd is not None:
            e = np.abs(sol.astype(LD) - xr).max(axis=2) / np.abs(xr).max(axis=2)
            if fwd == "tight":
                _report(mode, "forward", e[good].max())
                assert e[good].max() <= 1e-13, (tag, e[good].max(), np.argwhere(good & (e > 1e-13))[:8])
            else:
                kap = ref["cond"].reshape(B, K)
                lim = 64 * U * kap if fwd == "cond" else np.maximum(1e-13, 64 * U * kap)
                _report(mode, "forward", e[good].max())
                _report(mode, "forward/(u kappa)", (e[good] / (U * kap[good])).max())
                assert np.all(e[good] <= lim[good]), (tag, np.argwhere(good & (e > lim))[:8])
    # 3. k_solve_warp is bit-identical to k_solve_tpb (NaN patterns of the untouched rows included)
    dx1, ok1, lu1 = res[1]
    assert np.array_equal(dx1.view(np.uint64), dx0.view(np.uint64)), name
    assert np.array_equal(ok1, ok0) and np.array_equal(lu1.view(np.uint64), lu0.view(np.uint64)), name
    return res, ref, lam_k


def _random_batch(rng, ns, n_cap, pad=np.nan, **kw):
    Hb = np.zeros((len(ns), 4 * n_cap, 12))
    for i, n in enumerate(ns):
        A, b = spd_real_block(rng, 1, int(n), **kw)
        Hb[i] = embed(A, b, int(n), n_cap, pad=pad)[0]
    return Hb


SMALL_N = list(range(3, 73))
LARGE_N = [115, 116, 117, 145, 199, 200, 201, 255, 256, 257, 383, 384, 385, 510, 511, 512]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 6])
def test_random_spd_every_small_n(gpu, K):
    """class (a), every n in 3 .. 72 (every n mod 16, nblk 0 / 1 / 2 of k_solve_lat, every 4n mod 11 of k_solve_tpb),
    ragged: n < n_cap; 70 bands x K trials is not a multiple of 32"""
    rng = np.random.default_rng(K)
    ns = SMALL_N if K == 6 else SMALL_N[::-1][:69]
    Hb = _random_batch(rng, ns, 75)
    lam0 = rng.uniform(1e-4, 1e-1, len(ns))
    _check(gpu, Hb, ns, lam0, 2.0, K, fwd="tight", name=f"small K={K}")


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 8])
def test_random_spd_large_n(gpu, K):
    """class (a) at the large shapes, n_cap = 512 (n = 512 = n_cap included), 17 bands"""
    rng = np.random.default_rng(10 + K)
    ns = LARGE_N + [300]
    Hb = _random_batch(rng, ns, 512)
    _check(gpu, Hb, ns, rng.uniform(1e-3, 1.0, len(ns)), 2.0, K, fwd="tight", name=f"large K={K}")


@pytest.mark.gpu
def test_full_capacity_batch(gpu):
    """n = n_cap = 512 for every band (no padding rows at all; k_solve_lat at 196 KB of shared memory)"""
    rng = np.random.default_rng(99)
    Hb = _random_batch(rng, [512] * 3, 512)
    _check(gpu, Hb, 512, [1e-3, 0.1, 3.0], 2.0, 6, fwd="tight", name="n=n_cap=512")


@pytest.mark.gpu
def test_padding_is_never_read(gpu):
    """NaN or zeros after row 4n of every band: bit-identical results"""
    rng = np.random.default_rng(4)
    ns = [3, 16, 17, 31, 47, 63, 64, 65, 100, 250, 500]
    r1 = _random_batch(np.random.default_rng(4), ns, 511, pad=np.nan)
    r2 = _random_batch(np.random.default_rng(4), ns, 511, pad=0.0)
    lam0 = rng.uniform(1e-3, 1e-1, len(ns))
    a, _, _ = _check(gpu, r1, ns, lam0, 2.0, 6, fwd="tight", name="pad nan")
    b = _run_modes(gpu, r2, np.array(ns, np.int32), lam0, np.full(len(ns), 2.0), 6)
    for mode in MODES:
        inside = np.arange(4 * 511)[None, None, :] < 4 * np.array(ns)[:, None, None]
        assert np.array_equal(np.where(inside, a[mode][0], 0).view(np.uint64), np.where(inside, b[mode][0], 0).view(np.uint64)), mode
        assert np.array_equal(a[mode][1], b[mode][1]) and np.array_equal(a[mode][2], b[mode][2]), mode


@pytest.mark.gpu
@pytest.mark.parametrize("scenario", ["C1", "C2", "C3", "C4", "holonomic", "shapes_polygon"])
def test_kernel_a_systems(gpu, scenario):
    """class (b): the systems kernel A builds, at outer iterations 0 and 3; lambda_0 = 1e-5 max real diagonal
    (computeLambdaInit), escalated with ni = 2 over K = 8 trials - one complete first round of an LM iteration.
    The first trials of these systems are not well conditioned (kappa up to ~1e5 .. 1e6 at lambda_0): the forward
    error is held to 1e-13 or, where that is below what any backward-stable solve guarantees, to 64 u kappa"""
    import teb_local_planner_b200 as T
    from tests import scenarios
    p, hb = scenarios.scenario(scenario, candidates=5)
    g = T.TebGpu(hb.B, hb.n_cap, hb.S, max(hb.M_cap, 1), hb.V_cap, max_obst_vertices=hb.PV_cap)
    g.set_params(p)
    systems = []
    for outer in (0, 3):
        Hb, _ = g.build_system(hb, outer)
        systems.append(Hb)
    g.close()
    Hb = np.concatenate(systems)
    ns = np.concatenate([hb.n, hb.n]).astype(np.int32)
    for b in range(len(ns)):
        Hb[b, 4 * ns[b]:] = np.nan
    real = np.stack([row_is_real(Hb.shape[1], int(v)) for v in ns])
    lam0 = 1e-5 * np.where(real, np.abs(Hb[:, :, 0]), 0).max(axis=1)
    assert (len(ns) * 8) % 32 != 0
    if Hb.shape[1] > 4 * 512 or len(ns) > 128:
        pytest.skip("scenario larger than the solve context")
    _, ref, _ = _check(gpu, Hb, ns, lam0, 2.0, 8, fwd="tight_or_cond", name=scenario)
    print(f"{scenario}: condition estimates {np.nanmin(ref['cond']):.1e} .. {np.nanmax(ref['cond']):.1e}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["graded", "rank_deficient"])
def test_ill_conditioned(gpu, kind):
    """class (c): kappa up to ~1e12 .. 1e14 with a tiny damping; forward error within 64 u kappa"""
    rng = np.random.default_rng(21 if kind == "graded" else 22)
    ns = [5, 17, 33, 64, 97, 200, 257]
    Hb = np.zeros((len(ns), 4 * 260, 12))
    for i, n in enumerate(ns):
        if kind == "graded":
            A, b = spd_real_block(rng, 1, n, ridge=0.05)
            A, b = graded(A, b, rng, span=6.0)
        else:
            A, b = spd_real_block(rng, 1, n, ridge=0.0, rank_drop=7)
            A[:, :, 0] += 1e-12 * A[:, :, 0].max()
        Hb[i] = embed(A, b, n, 260)[0]
    real = np.stack([row_is_real(Hb.shape[1], v) for v in ns])
    dmax = np.where(real, np.abs(np.nan_to_num(Hb[:, :, 0])), 0).max(axis=1)
    _, ref, _ = _check(gpu, Hb, ns, 1e-14 * dmax, 2.0, 6, fwd="cond", name=kind)
    kap = ref["cond"][np.isfinite(ref["cond"])]
    print(f"{kind}: condition estimates {kap.min():.1e} .. {kap.max():.1e}")
    assert kap.max() >= 1e10, "the class is meant to be ill-conditioned"


@pytest.mark.gpu
@pytest.mark.parametrize("e", [-200, 200])
def test_power_of_two_rescaling_is_exact(gpu, e):
    """class (c): H, b and lambda scaled by 2^e - every operation of the three solvers scales exactly, so the solution,
    the flags and everything else are bit for bit those of the unscaled system"""
    rng = np.random.default_rng(31)
    ns = [3, 19, 40, 129, 300]
    Hb = _random_batch(rng, ns, 300)
    lam0 = rng.uniform(1e-3, 1e-1, len(ns))
    base = _run_modes(gpu, Hb, np.array(ns, np.int32), lam0, np.full(len(ns), 2.0), 6)
    Hs = Hb * 2.0 ** e
    for i, n in enumerate(ns):
        Hs[i, :4 * n, 0] = np.where(row_is_real(4 * n, n), Hs[i, :4 * n, 0], 1.0)
    res, _, _ = _check(gpu, Hs, ns, lam0 * 2.0 ** e, 2.0, 6, fwd="tight", name=f"2^{e}")
    for mode in MODES:
        assert np.array_equal(res[mode][0].view(np.uint64), base[mode][0].view(np.uint64)), mode
        assert np.array_equal(res[mode][1], base[mode][1]), mode


@pytest.mark.gpu
def test_indefinite_systems_escalate_to_the_first_positive_definite_trial(gpu):
    """class (d): real block with smallest eigenvalue -mu; trial k is positive definite iff lambda_k > mu. mu / lambda_0
    is chosen away from every lambda_k / lambda_0 (1, 2, 8, 64, 1024, ...) by far more than 1 %"""
    rng = np.random.default_rng(41)
    ns = [3, 4, 11, 16, 17, 29, 48, 70, 131, 256, 400]
    ratios = [0.3, 1.5, 5.0, 20.0, 100.0, 700.0, 3.0, 40.0, 0.5, 12.0, 300.0]
    K = 8
    Hb = np.zeros((len(ns), 4 * 400, 12))
    lam0 = np.zeros(len(ns))
    for i, (n, ratio) in enumerate(zip(ns, ratios)):
        A, b = spd_real_block(rng, 1, n, ridge=0.05)
        Nr = 4 * n - 7
        ab = np.zeros((BW + 1, Nr))
        for k in range(min(BW, Nr - 1) + 1):
            ab[k, :Nr - k] = A[0, k:, k]
        emin = scipy.linalg.eigvals_banded(ab, lower=True, select="i", select_range=(0, 0))[0]
        mu = 0.1 * A[0, :, 0].mean()
        A[0, :, 0] -= emin + mu
        lam0[i] = mu / ratio
        Hb[i] = embed(A, b, n, 400)[0]
    lk = host_lambdas(lam0, 2.0, K)
    mu = lam0 * np.array(ratios)
    assert np.all(np.abs(lk / mu[:, None] - 1) > 0.01)
    res, ref, _ = _check(gpu, Hb, ns, lam0, 2.0, K, fwd=None, name="indefinite")
    want_first = (lk > mu[:, None]).argmax(axis=1)
    ref_first = ref["all_pivots_positive"].reshape(len(ns), K).argmax(axis=1)
    assert np.array_equal(ref_first, want_first)
    for mode in MODES:
        ok = res[mode][1].astype(bool)
        assert np.array_equal(ok.argmax(axis=1), want_first), (mode, ok.argmax(axis=1), want_first)
        assert np.all(ok == (lk > mu[:, None])), mode


@pytest.mark.gpu
def test_failure_contract_edges(gpu):
    """pivot_ok (teb_spec.cuh) in every mapping: a zero or a subnormal pivot fails; a solution that overflows from valid
    pivots does not (CSparse reports success, the non-finite chi2 ends the LM iteration as in g2o)"""
    n = 6
    rng = np.random.default_rng(51)
    A, b = spd_real_block(rng, 1, n)
    Nr = 4 * n - 7
    cases = []
    for dpiv, bval, want in ((0.0, 1.0, False),          # exact zero pivot
                             (1e-310, 1.0, False),       # subnormal pivot
                             (1e-300, 1e300, True)):     # valid pivots, x_7 = 1e300 / 1e-300 overflows
        Ad = np.zeros_like(A)
        Ad[0, :, 0] = 1.0
        Ad[0, 7, 0] = dpiv
        bd = b.copy()
        bd[0, 7] = bval
        cases.append((Ad, bd, want))
    Hb = np.concatenate([embed(a, bb, n, n) for a, bb, _ in cases])
    res = _run_modes(gpu, Hb, np.full(len(cases), n, np.int32), np.zeros(len(cases)), np.full(len(cases), 2.0), 3)
    want = np.array([w for _, _, w in cases])
    for mode in MODES:
        ok = res[mode][1]
        assert np.all(ok == want[:, None]), (mode, ok)
        assert not np.isfinite(res[mode][0][2, :, :4 * n]).all(axis=1).any(), mode
