"""Pins the oracle restatement (oracle/teb_oracle.c) against the REFERENCE'S OWN CODE: oracle/_ref/libteb_ref.so is
src/optimal_planner.cpp + src/timed_elastic_band.cpp + src/obstacles.cpp and their headers compiled where they lie,
with stand-ins only for the absent third-party code (Eigen, boost, ROS messages, the g2o optimizer; oracle/ref_shims/).

What is compared: TebConfig() defaults, penalties.h, every footprint x obstacle distance, the graph buildGraph() builds
edge by edge (errors, information, Jacobians incl. the two analytic overrides), H / b / chi2, whole optimizeTEB calls
(poses, n, cost, number of LM trials), computeCurrentCost outside optimizeTEB, autoResize, initTrajectoryToGoal,
updateAndPruneTEB. The bar is BIT EQUALITY (both sides are fp64, compiled without FMA contraction); where a libm call
order differs the tolerance is written at the assertion.

The reference's side of every comparison is read from tests/golden/golden_pin_v1.npz (`ref_binding.Pins`), recorded
from the library by tests/golden/make_golden_pin.py: the values where a tolerance applies, a digest of the result where
the bar is bit equality."""
import ctypes as C
import functools
import os

import numpy as np
import pytest

from teb_local_planner_b200 import abi, scenes
from tests import ref_binding as rb
from tests import scenarios
from tests.ref_binding import pins  # noqa: F401  (fixture)

GOLDEN_REF = os.path.join(os.path.dirname(__file__), "golden", "golden_ref_v1.npz")


def test_default_params_are_the_reference_constructor_defaults(teblib, pins):
    names = [name for name, _ in abi.TebParams._fields_ if not name.startswith("_")]
    field = lambda q, name: list(getattr(q, name)) if isinstance(getattr(q, name), C.Array) else getattr(q, name)
    ref = pins.value(lambda: [np.array(field(rb.default_params(), name)) for name in names])
    mine = abi.default_params()
    lib = abi.TebParams()
    teblib.tebgpu_default_params(C.byref(lib))
    for name, a in zip(names, ref):
        assert np.array_equal(a, field(mine, name)) and np.array_equal(a, field(lib, name)), name


def test_penalties_bit_equal(oracle, pins):
    L = oracle.lib()
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.normal(0, 1, 4000), [0.0, 0.35, -0.35, 0.4, -0.4, 0.45, 0.05, -0.05, 0.5, 0.55, 0.6]])
    for a, eps in ((0.4, 0.05), (0.3, 0.0), (0.5, 0.05)):
        pins.equal(lambda: [[rb.penalty(0, v, a, 0.0, eps), rb.penalty(1, v, -0.2, a, eps), rb.penalty(2, v, a, 0.0, eps)] for v in vals],
                   [[L.teb_oracle_penalty_interval(v, a, eps), L.teb_oracle_penalty_interval2(v, -0.2, a, eps),
                     L.teb_oracle_penalty_below(v, a, eps)] for v in vals], (a, eps))


@pytest.mark.parametrize("footprint", ["point", "circular", "two_circles", "line", "polygon"])
def test_distances_every_footprint_and_obstacle_type(oracle, pins, footprint):
    p, hb = scenarios.scenario("shapes_" + footprint, candidates=2)
    obst = hb.obstacles[0][:hb.obst_count[0]]
    kinds = set(int(o["type"]) for o in obst)
    assert kinds >= {abi.TEB_OBST_POINT, abi.TEB_OBST_LINE, abi.TEB_OBST_PILL, abi.TEB_OBST_POLYGON}
    circ = obst[0].copy()
    circ["type"], circ["radius"] = abi.TEB_OBST_CIRCULAR, 0.3
    rng = np.random.default_rng(5)
    queries = []
    for o in list(obst) + [circ]:
        if not o["dynamic"]:            # a static obstacle has no velocity in the reference (obstacles.h:206 sets both)
            o = o.copy()
            o["vx"], o["vy"] = 0.0, 0.0
        for _ in range(12):
            pose = np.array([o["x"] + rng.normal(0, 1.0), o["y"] + rng.normal(0, 1.0), rng.uniform(-np.pi, np.pi)])
            queries += [(pose, o, t) for t in (None, 0.0, 1.7)]
    d_ref = pins.value(lambda: [rb.distance(p, pose, o, hb.obst_vertices[0], t) for pose, o, t in queries])
    d_orc = [oracle.distance(p, pose, o, hb.obst_vertices[0], 0.0 if t is None else t) if (t is not None) else
             _static_distance(oracle, p, pose, o, hb.obst_vertices[0]) for pose, o, t in queries]
    worst = np.abs(np.array(d_ref) - np.array(d_orc)).max()
    assert worst <= 1e-15, worst


def _static_distance(oracle, p, pose, o, verts):
    """calculateDistance ignores the obstacle's velocity: evaluate the oracle on a static copy"""
    s = o.copy()
    s["dynamic"], s["vx"], s["vy"] = 0, 0.0, 0.0
    return oracle.distance(p, pose, s, verts, 0.0)


@pytest.mark.parametrize("name", scenarios.ALL)
def test_graph_edges_and_normal_equations_bit_equal(oracle, pins, name):
    """buildGraph + computeActiveErrors + buildSystem: every active edge (dimension, vertex ids, error, information,
    Jacobian) and the assembled H / b / chi2, for obstacle weight multipliers 1 and 4"""
    p, hb = scenarios.scenario(name)
    for b in range(hb.B):
        n = int(hb.n[b])
        kw = scenarios.band_kwargs(hb, b)
        for wm in (1.0, 4.0):
            Ho, bo, co = oracle.build_system(p, hb.poses[b], n, weight_multiplier=wm, jac_mode=oracle.JAC_G2O, **kw)
            eo = oracle.dump_edges(p, hb.poses[b], n, weight_multiplier=wm, jac_mode=oracle.JAC_G2O, **kw)
            ref = functools.cache(lambda: rb.build_system(p, hb.poses[b], n, weight_multiplier=wm, want_edges=True, **kw))
            pins.equal(lambda: ref()[3][:, :8], eo[:, :8], (name, b, wm, "errors / information"))
            pins.equal(lambda: ref()[3][:, 53:], eo[:, 53:], (name, b, wm, "graph structure"))
            pins.equal(lambda: ref()[3], eo, (name, b, wm, "Jacobians"))
            pins.equal(lambda: ref()[:3], (Ho, bo, co), (name, b, wm, "H / b / chi2"))


@pytest.mark.parametrize("name", scenarios.ALL)
def test_optimize_teb_bit_equal(oracle, pins, name):
    """whole optimizeTEB calls (outer x inner LM iterations, autoResize, weight adaptation, cost): poses, n, cost and
    the number of LM trials of the reference's code and of the restatement are identical"""
    p, hb = scenarios.scenario(name)
    args = abi.make_args(p.no_inner_iterations, p.no_outer_iterations, True, p.selection_obst_cost_scale,
                         p.selection_viapoint_cost_scale, False)
    for b in range(hb.B):
        n = int(hb.n[b])
        kw = scenarios.band_kwargs(hb, b)
        ro, co, so = oracle.optimize_band(p, hb.poses[b], n, args=args, jac_mode=oracle.JAC_G2O, n_cap=hb.n_cap, **kw)
        pins.equal(lambda: _optimized(rb.optimize_band(p, hb.poses[b], n, args=args, n_cap=hb.n_cap, **kw)),
                   (True, ro, co, so.lm_trials, so.rejected, bool(so.status & abi.TEB_STATUS_TERMINATED)), (name, b))


def _optimized(res):
    """the parts of the reference's optimizeTEB result the oracle's must equal: ok, band, cost, LM trials / rejections,
    termination"""
    rr, cr, sr, ok = res
    return ok, rr, cr, sr["lm_trials"], sr["rejected"], sr["terminated"]


def test_optimize_teb_alternative_time_cost_and_disabled(oracle, pins):
    p, hb = scenarios.scenario("C2")
    kw = scenarios.band_kwargs(hb, 0)
    args = abi.make_args(3, 2, True, 7.0, 3.0, True)
    ro, co, so = oracle.optimize_band(p, hb.poses[0], int(hb.n[0]), args=args, jac_mode=oracle.JAC_G2O, **kw)
    ok_band_cost = lambda r: (r[3], r[0], r[1])
    pins.equal(lambda: ok_band_cost(rb.optimize_band(p, hb.poses[0], int(hb.n[0]), args=args, **kw)), (True, ro, co))
    p.optimization_activate = 0        # optimizeTEB returns false before touching anything (optimal_planner.cpp:185)
    ro, co, so = oracle.optimize_band(p, hb.poses[0], int(hb.n[0]), args=args, jac_mode=oracle.JAC_G2O, **kw)
    # (isOptimized() is not checked: the constructor used here leaves optimized_ uninitialised, optimal_planner.cpp:67-70)
    pins.equal(lambda: ok_band_cost(rb.optimize_band(p, hb.poses[0], int(hb.n[0]), args=args, **kw))[:2],
               (False, hb.poses[0][:hb.n[0]]))
    assert np.array_equal(ro, hb.poses[0][:hb.n[0]])
    assert not (so.status & abi.TEB_STATUS_OPTIMIZED)


def test_divergence_detection_matches(oracle, pins):
    """hasDiverged (optimal_planner.cpp:1023-1039): chi2 of the final state vs divergence_detection_max_chi_squared"""
    p, hb = scenarios.scenario("divergence")
    args = abi.make_args(5, 4, True, 100.0, 1.0, False)
    seen = set()
    for thr in (10, 100000):
        p.divergence_detection_max_chi_squared = thr
        for b in range(hb.B):
            kw = scenarios.band_kwargs(hb, b)
            ro, co, so = oracle.optimize_band(p, hb.poses[b], int(hb.n[b]), args=args, jac_mode=oracle.JAC_G2O, **kw)
            ref = functools.cache(lambda: rb.optimize_band(p, hb.poses[b], int(hb.n[b]), args=args, **kw))
            pins.equal(lambda: ref()[:2], (ro, co), (thr, b))
            diverged = bool(pins.value(lambda: ref()[2]["diverged"])[0])
            assert diverged == (so.chi2_final > thr)
            seen.add(diverged)
    assert seen == {True, False}


def test_compute_cost_outside_optimize_is_undefined_in_the_reference(oracle, pins):
    """computeCurrentCost on a FRESH graph (optimal_planner.cpp:1045-1051, the path HomotopyClassPlanner::
    computeCurrentCost takes): buildGraph + initializeOptimization never evaluate an edge and computeInitialGuess does
    nothing for TEB edges, so edge->chi2() reads the `_error` members as constructed. Upstream g2o leaves them
    uninitialised (Eigen does not zero): the reference's value is undefined. With the zero-initialising stand-in the
    reference code returns exactly 0 (only the alternative time cost survives) - which documents that nothing on that
    path computes errors. tebgpu_compute_cost defines the call as the scaled chi2 AT the current state instead
    (DESIGN.md); that value is what the restatement below computes, and the GPU test checks the C-ABI against it."""
    p, hb = scenarios.scenario("C2")
    kw = scenarios.band_kwargs(hb, 0)
    n = int(hb.n[0])
    plain, alt = pins.value(lambda: [rb.compute_cost(p, hb.poses[0], n, args=abi.make_args(5, 4, True, 50.0, 2.5, alt_time), **kw)
                                     for alt_time in (False, True)])
    assert plain == 0.0
    t = 0.0
    for i in range(n - 1):              # getSumOfAllTimeDiffs (timed_elastic_band.cpp:184-192), same summation order
        t += hb.poses[0][i, 3]
    assert alt == t
    assert _cost_from_oracle(oracle, p, hb, 0, abi.make_args(5, 4, True, 50.0, 2.5, False)) > 0


def _cost_from_oracle(oracle, p, hb, b, args):
    """scaled chi2 by family at the current state: chi2 is linear in the information weights and a zero weight removes
    the family's edges (optimal_planner.cpp:337, :342, :677), so differences of three oracle builds isolate the families"""
    kw = scenarios.band_kwargs(hb, b)
    n = int(hb.n[b])

    def chi(q):
        return oracle.build_system(q, hb.poses[b], n, jac_mode=oracle.JAC_G2O, **kw)[2]
    base = chi(p)
    q = type(p).from_buffer_copy(p)
    q.weight_obstacle, q.weight_inflation, q.weight_dynamic_obstacle, q.weight_dynamic_obstacle_inflation = 0, 0, 0, 0
    obst = base - chi(q)
    q = type(p).from_buffer_copy(p)
    q.weight_viapoint = 0
    via = base - chi(q)
    return args.obst_cost_scale * obst + args.viapoint_cost_scale * via + (base - obst - via)


@pytest.mark.parametrize("case", ["large_at_end", "small_at_end", "middle_and_end"])
def test_autoresize_reference_gtests_on_reference_code(oracle, teblib, pins, case):
    """test/teb_basics.cpp:5-68 (the reference's own gtests): same inputs, same assertions, executed on the reference's
    TimedElasticBand; the restatement and the product's host routine must return the identical band"""
    dt, hyst = 0.1, 0.1 / 3.0
    dts = [dt] * 9
    if case == "large_at_end":
        dts.append(dt + 2 * hyst)
    elif case == "small_at_end":
        dts.append(dt - 2 * hyst)
    else:
        dts[5] = dt + 2 * hyst
        dts.append(dt - 2 * hyst)
    n = len(dts) + 1
    rec = np.zeros((64, 4))
    rec[:n, 0] = np.arange(n)
    rec[:n - 1, 3] = dts
    out = pins.value(lambda: rb.auto_resize(rec, n, dt, hyst, 3, 100, False, n_cap=64))[0]
    d = out[:-1, 3]
    assert np.all(d <= dt + hyst + 1e-3) and np.all(dt - hyst - 1e-3 <= d)     # ASSERT_LE pairs of the gtest
    assert np.array_equal(out, oracle.auto_resize(rec, n, dt, hyst, 3, 100, False, n_cap=64))
    mine = rec.copy()
    nn = teblib.tebgpu_auto_resize_host(mine.ctypes.data, n, 64, dt, hyst, 3, 100, 0)
    assert nn == len(out) and np.array_equal(mine[:nn], out)


def test_autoresize_random_bit_equal(oracle, pins):
    rng = np.random.default_rng(2)
    for k in range(300):
        n = int(rng.integers(3, 40))
        rec = np.zeros((n, 4))
        rec[:, 0] = np.cumsum(rng.uniform(0.0, 0.3, n))
        rec[:, 1] = rng.normal(0, 0.5, n)
        rec[:, 2] = rng.uniform(-3.2, 3.2, n)
        rec[:n - 1, 3] = rng.choice([0.05, 0.1, 0.29, 0.3, 0.41, 0.8, 1.5], n - 1) * rng.uniform(0.9, 1.1, n - 1)
        fast = bool(k % 2)
        mn = int(rng.integers(3, 6)) if k % 3 else 3
        mx = int(rng.choice([12, 50, 500]))
        c = oracle.auto_resize(rec, n, 0.3, 0.1, mn, mx, fast, n_cap=1024)
        pins.equal(lambda: rb.auto_resize(rec, n, 0.3, 0.1, mn, mx, fast, n_cap=1024), c, k)


def test_init_trajectory_bit_equal(oracle, pins):
    rng = np.random.default_rng(4)
    for k in range(100):
        start = np.array([rng.normal(0, 2), rng.normal(0, 2), rng.uniform(-3, 3)])
        goal = start + np.array([rng.normal(0, 3), rng.normal(0, 3), rng.uniform(-1, 1)])
        diststep = float(rng.choice([0.0, 0.1, 0.35]))
        back = bool(k % 4 == 0)
        ms = int(rng.integers(3, 8)) if k % 2 else 3
        c = oracle.init_trajectory(start, goal, diststep, 0.4, ms, back, n_cap=2048)
        pins.equal(lambda: rb.init_trajectory(start, goal, diststep, 0.4, ms, back, n_cap=2048), c, k)


def test_golden_reference_vectors_are_current(pins):
    """the committed fixture was generated from the reference build the other pins come from: a slice regenerated from
    that build equals the fixture"""
    from tests.golden import make_golden_ref
    z = np.load(GOLDEN_REF, allow_pickle=False)
    only = ("C1", "via_ordered")
    keys = [k for k in z.files if k.split("/")[0] in only]

    def fresh():
        f = make_golden_ref.generate(only=only)
        assert sorted(f) == sorted(keys)
        return [f[k] for k in keys]
    pins.equal(fresh, [z[k] for k in keys])


@pytest.mark.parametrize("cfg", ["C1", "C2", "C3", "C4"])
def test_h_signatures_match_the_reference_header(oracle, pins, cfg):
    """calculateEquivalenceClass executed by the reference's own h_signature.h (HSignature: long double complex
    accumulation; HSignature3d: numeric integration over the x-y-t obstacle 'conductors', with and without the band's
    time differences) against the oracle restatement, plus isValid / isReasonable and the class comparison the planner
    derives from them. 2-D: relative 1e-15 of the long double result; 3-D: bit equal."""
    from tests.golden import make_golden
    p, hb = scenes.make_config_batch(cfg, candidates=6, seed=17)
    obst = hb.obstacles[0][:hb.obst_count[0]]
    sig2 = []
    for b in range(hb.B):
        rec, n = hb.poses[b], int(hb.n[b])
        p.include_dynamic_obstacles = 0
        want, valid, reasonable = pins.value(lambda: rb.h_signature(p, rec, n, obst))
        want = complex(*want)
        got = oracle.h_signature(p, rec, n, obst)
        assert valid and np.isfinite(want.real) and np.isfinite(want.imag)
        assert abs(got - want) <= 1e-15 * max(1.0, abs(want)), (cfg, b, got, want)
        sig2.append((got, want))
        p.include_dynamic_obstacles = 1
        for use_dt in (True, False):
            want3, valid3, reasonable3 = pins.value(lambda: rb.h_signature(p, rec, n, obst, use_timediffs=use_dt))
            got3 = oracle.h_signature(p, rec, n, obst, use_timediffs=use_dt)
            assert valid3
            assert np.array_equal(got3, want3), (cfg, b, use_dt, np.abs(got3 - want3).max())
            assert reasonable3 == bool(np.all(want3 <= 1.0))
    # HSignature::isEqual (h_signature.h:195-206): both parts within h_signature_threshold - same partition either way
    thr = p.h_signature_threshold
    eq = lambda x, y: abs(x.real - y.real) <= thr and abs(x.imag - y.imag) <= thr
    for i in range(hb.B):
        for j in range(hb.B):
            assert eq(sig2[i][0], sig2[j][0]) == eq(sig2[i][1], sig2[j][1])
    # the committed H-signature fixtures (tests/golden/golden_v2.npz) agree with the reference header as well
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_v2.npz"), allow_pickle=False)
    for name, pp, hbb in make_golden.hsig_cases():
        ob = hbb.obstacles[0][:hbb.obst_count[0]]
        for b in range(hbb.B):
            want = pins.value(lambda: rb.h_signature(pp, hbb.poses[b], hbb.n[b], ob))[0]
            have = g[name][b]
            if pp.include_dynamic_obstacles:
                assert np.array_equal(want, have[:len(ob)])
            else:
                want = complex(*want)
                assert abs(want - complex(have[0], have[1])) <= 1e-15 * max(1.0, abs(want))


def _explorer_inputs(rng, n_obst, dynamic):
    from oracle import hcp_explore as X
    rows = np.zeros(n_obst, abi.OBST_DTYPE)
    obstacles, pool = [], []
    for m in range(n_obst):
        kind = ["point", "circle", "line"][int(rng.integers(3))]
        c = np.array([rng.uniform(-3.2, 3.2), rng.uniform(-1.6, 1.6)])
        if kind == "point":
            rows[m]["type"], rows[m]["x"], rows[m]["y"] = abi.TEB_OBST_POINT, c[0], c[1]
            obstacles.append(X.Obst("point", tuple(c)))
        elif kind == "circle":
            r = rng.uniform(0.1, 0.4)
            rows[m]["type"], rows[m]["x"], rows[m]["y"], rows[m]["radius"] = abi.TEB_OBST_CIRCULAR, c[0], c[1], r
            obstacles.append(X.Obst("circle", tuple(c), r))
        else:
            d = rng.normal(0, 0.35, 2)
            a, b = c - d, c + d
            rows[m]["type"], rows[m]["vertex_begin"], rows[m]["vertex_count"] = abi.TEB_OBST_LINE, len(pool), 2
            pool += [a, b]
            ctr = 0.5 * (a + b)
            rows[m]["x"], rows[m]["y"] = ctr[0], ctr[1]
            obstacles.append(X.Obst("line", tuple(ctr), vertices=[tuple(a), tuple(b)]))
        if dynamic and rng.random() < 0.4:
            rows[m]["vx"], rows[m]["vy"], rows[m]["dynamic"] = rng.normal(0, 0.1), rng.normal(0, 0.1), 1
    return rows, obstacles, (np.array(pool) if pool else None)


@pytest.mark.parametrize("prm", [False, True])
@pytest.mark.parametrize("dynamic", [0, 1])
def test_candidate_exploration_matches_the_reference_planner(oracle, pins, prm, dynamic):
    """exploreEquivalenceClassesAndInitTebs of the reference's own HomotopyClassPlanner / graph_search.cpp (key-point graph
    and probabilistic roadmap, DepthFirst enumeration order, addAndInitNewTeb with the path variant of
    initTrajectoryToGoal, H-signature filtering with both signature kinds, class budget) against the sequential
    restatement oracle/hcp_explore.py - the one the GPU test of the drop-in planner is compared with. Same candidates, same
    order, initial bands equal to 1e-12 (the restatement evaluates atan2 / hypot in Python). The roadmap's random stream is
    boost's (absent from the image): both sides restate the same published generator, so that part pins consistency only."""
    from oracle import hcp_explore as X
    rng = np.random.default_rng(100 + 2 * int(prm) + dynamic)
    for case in range(12):
        p = abi.default_params()
        p.include_dynamic_obstacles = dynamic
        rows, obstacles, pool = _explorer_inputs(rng, int(rng.integers(2, 7)), dynamic)
        hcp = {"max_number_classes": int(rng.integers(2, 8)), "obstacle_heading_threshold": [0.0, 0.45, 0.7][int(rng.integers(3))],
               "roadmap_graph_area_width": rng.uniform(3, 7), "roadmap_graph_area_length_scale": [1.0, 0.8][int(rng.integers(2))],
               "roadmap_graph_no_samples": int(rng.integers(5, 16))}
        start = [-4.0, rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.4)]
        goal = [4.0, rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.4)]
        cycles = 2
        counts, *bands = pins.value(lambda: _flat_explore(rb.hcp_explore(p, hcp, start, goal, rows, pool, cycles=cycles, prm=prm)))
        ends = np.cumsum(counts).astype(int)
        want = [bands[e - int(k):e] for k, e in zip(counts, ends)]
        ex = X.Explorer(p, hcp, oracle, rows, obstacles)
        for c in range(cycles):
            ex.classes, ex.tebs = [], []
            (ex.prob_roadmap_graph if prm else ex.lr_key_point_graph)(start, goal, p.min_obstacle_dist)
            assert len(ex.tebs) == len(want[c]), (case, c, len(ex.tebs), len(want[c]))
            for k, (got, ref) in enumerate(zip(ex.tebs, want[c])):
                assert got.shape == ref.shape, (case, c, k, got.shape, ref.shape)
                assert np.abs(got - ref).max() < 1e-12, (case, c, k, np.abs(got - ref).max())


def _flat_explore(res):
    """hcp_explore's result (per cycle a list of bands) as [candidates per cycle, band, band, ...]"""
    return [np.array([len(c) for c in res])] + [band for c in res for band in c]


def _flat_plan(res):
    """hcp_plan's result as ([(ok, best, candidates), costs] per cycle, [band, band, ...])"""
    return ([x for ok, best, cands in res for x in (np.array([ok, best, len(cands)]), np.array([c for c, _ in cands]))],
            [band for _, _, cands in res for _, band in cands])


def _unflat_plan(heads, bands):
    res = []
    for (ok, best, k), costs in zip(heads[0::2], heads[1::2]):
        res.append((bool(ok), int(best), list(zip(costs.tolist(), bands[:int(k)]))))
        bands = bands[int(k):]
    return res


@pytest.mark.parametrize("prm", [False, True])
def test_planning_cycles_match_the_reference_planner(oracle, teblib, pins, prm):
    """consecutive HomotopyClassPlanner::plan(start, goal) calls of the reference's own planner (updateAllTEBs,
    renewAndAnalyzeOldTebs, deletePlansDetouringBackwards, graph exploration, optimizeAllTEBs, selectBestTeb) against the
    sequential restatement oracle/hcp_explore.py::Planner with the start pose moving along: same number of candidates,
    same order, same pose counts, same selected candidate in every cycle. The reference optimises with numeric Jacobians
    (the restatement is switched to that mode); initial bands that differ in the last bit (Python vs C atan2 / hypot) come
    out ~1e-7 apart after 20 LM iterations, hence 1e-5 on poses and 1e-6 relative on costs.
    The reference's TebConfig constructor leaves hcp.max_number_plans_in_current_class uninitialised (candidate counts
    varied from process to process until oracle/ref_driver.cpp set the dynamic_reconfigure default 1)."""
    from oracle import hcp_explore as X
    rng = np.random.default_rng(300 + int(prm))
    for case in range(5):
        p = abi.default_params()
        p.include_dynamic_obstacles = 0
        p.selection_cost_hysteresis = [1.0, 0.9, 0.8][case % 3]
        carried_best = False
        rows, obstacles, pool = _explorer_inputs(rng, int(rng.integers(2, 5)), 0)
        hcp = {"max_number_classes": int(rng.integers(2, 5)), "obstacle_heading_threshold": 0.45,
               "roadmap_graph_area_width": 5.0, "roadmap_graph_area_length_scale": 1.0, "roadmap_graph_no_samples": 10}
        goal = [4.0, rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2)]
        starts = [[-4.0 + 0.2 * c, 0.03 * c + rng.normal(0, 0.01), 0.05] for c in range(4)]
        ref = functools.cache(lambda: _flat_plan(rb.hcp_plan(p, hcp, starts, goal, rows, pool, prm=prm)))
        # the bands are stored in float32: the bound below leaves room for the rounding, so that it still holds against
        # the reference's float64 bands
        want = _unflat_plan(pins.value(lambda: ref()[0]), pins.value(lambda: ref()[1], np.float32))
        pl = X.Planner(p, hcp, oracle, rows, obstacles, simple_exploration=not prm)
        pl.jac_mode = oracle.JAC_G2O
        pl.obst_vertices = pool
        args = abi.make_args(p.no_inner_iterations, p.no_outer_iterations, True, p.selection_obst_cost_scale, p.selection_viapoint_cost_scale,
                             bool(p.selection_alternative_time_cost))
        for c, (ok, best, cands) in enumerate(want):
            got_best = pl.plan(starts[c], goal, args, abi)
            assert ok and len(pl.tebs) == len(cands), (case, c, len(pl.tebs), len(cands))
            assert (got_best if got_best is not None else -1) == best, (case, c, got_best, best)
            # tebgpu_select_best (the C-ABI's selectBestTeb, a pure host function) on the REFERENCE's own costs: the band the
            # planner carried over as its best one sits at index 0 after renewAndAnalyzeOldTebs
            costs_ref = np.array([x for x, _ in cands])
            last = 0 if (c > 0 and carried_best) else -1
            assert teblib.tebgpu_select_best(costs_ref.ctypes.data, len(costs_ref), last, -1, float(p.selection_cost_hysteresis),
                                             float(p.selection_prefer_initial_plan)) == best, (case, c)
            carried_best = best >= 0
            for k, ((cost, band), rec) in enumerate(zip(cands, pl.tebs)):
                assert band.shape == rec.shape, (case, c, k, band.shape, rec.shape)
                assert (np.abs(band - rec) + np.abs(band) * 2.0 ** -24).max() < 1e-5, (case, c, k, np.abs(band - rec).max())
                assert abs(cost - pl.costs[k]) <= 1e-6 * max(1.0, abs(cost)), (case, c, k, cost, pl.costs[k])
