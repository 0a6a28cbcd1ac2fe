"""The drop-in layer's band operations against the REFERENCE's own code, operation by operation, bit for bit.

oracle/_ref/libteb_ref.so (the reference's timed_elastic_band.cpp / optimal_planner.cpp compiled unmodified against
stand-in headers) and teb_local_planner_b200/host/test/libteb_host_pin.so (this repository's TimedElasticBand /
TebOptimalPlanner) expose the same operation codes (teb_ref_band_op / teb_host_band_op); both get the same random inputs.
Covers initTrajectoryToGoal (start / goal, plan, 2-D path of the graph search), updateAndPruneTEB,
findClosestTrajectoryPose, the time / distance sums, isTrajectoryInsideRegion, autoResize, getVelocityCommand,
getVelocityProfile and getFullTrajectory - the functions the round-1 review found lifted; they are rewritten and this is
what keeps them equal to the reference in behaviour. The reference's results are digests in tests/golden/golden_pin_v1.npz
(`ref_binding.Pins`), recorded from the library by tests/golden/make_golden_pin.py."""
import ctypes as C
import math
import os

import numpy as np
import pytest

from tests import ref_binding as rb
from tests.ref_binding import pins  # noqa: F401  (fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _band_op(fn):
    fn.restype = C.c_int32
    fn.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
    return fn


@pytest.fixture(scope="module")
def host():
    from teb_local_planner_b200 import build as b
    b.build()
    b.build_host()
    return _band_op(C.CDLL(b.HOST_PIN).teb_host_band_op)


@pytest.fixture
def ops(host, pins):
    def run(fn, op, rec, args, cap=8192):
        rec = None if rec is None else np.ascontiguousarray(rec, dtype=np.float64)
        a = np.ascontiguousarray(args, dtype=np.float64)
        out = np.full(cap, np.nan)
        k = fn(op, rec.ctypes.data if rec is not None else None, 0 if rec is None else len(rec), a.ctypes.data, len(a), out.ctypes.data, cap)
        assert k >= 0, (op, k)
        return out[:k].copy()

    def both(op, rec, args):
        h = run(host, op, rec, args)
        pins.equal(lambda: run(_band_op(rb.lib().teb_ref_band_op), op, rec, args), h, (op, args))
        return h

    return both


def _band(rng, n, wiggle=0.4):
    x = np.cumsum(rng.uniform(0.05, 0.3, n))
    y = np.cumsum(rng.normal(0, wiggle * 0.1, n))
    th = rng.uniform(-math.pi, math.pi, n) if rng.random() < 0.3 else np.arctan2(np.gradient(y), np.gradient(x)) + rng.normal(0, 0.05, n)
    dt = rng.uniform(0.05, 0.6, n)
    dt[-1] = 0
    return np.stack([x, y, th, dt], 1)


def test_init_from_start_and_goal(ops):
    rng = np.random.default_rng(1)
    for _ in range(200):
        s = [rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-math.pi, math.pi)]
        g = [rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(-math.pi, math.pi)]
        diststep = [0.0, 0.1, 0.25, 1.0][rng.integers(4)]
        out = ops(1, None, s + g + [diststep, rng.uniform(0.1, 1.0), int(rng.integers(2, 8)), int(rng.integers(2))])
        assert len(out) >= 8


def test_init_from_plan_and_from_path(ops):
    rng = np.random.default_rng(2)
    for _ in range(150):
        npts = int(rng.integers(2, 30))
        pts = np.cumsum(rng.normal(0.2, 0.3, (npts, 2)), 0)
        yaw = rng.uniform(-math.pi, math.pi, npts)
        plan = np.concatenate([pts, yaw[:, None]], 1).reshape(-1)
        ops(2, None, [rng.uniform(0.1, 1), rng.uniform(0.1, 1), int(rng.integers(2)), int(rng.integers(2, 40)), int(rng.integers(2)), npts] + plan.tolist())
        opt = lambda lo, hi: float("nan") if rng.random() < 0.4 else rng.uniform(lo, hi)
        ops(3, None, [rng.uniform(0.1, 1), rng.uniform(0.1, 1), opt(0.1, 1), opt(0.1, 1), opt(-3, 3), opt(-3, 3), int(rng.integers(2, 40)),
                      int(rng.integers(2)), npts] + pts.reshape(-1).tolist())


def test_update_and_prune_closest_pose_sums_region(ops):
    rng = np.random.default_rng(3)
    for _ in range(200):
        n = int(rng.integers(3, 60))
        rec = _band(rng, n)
        k = int(rng.integers(0, n))
        s = [rec[k, 0] + rng.normal(0, 0.1), rec[k, 1] + rng.normal(0, 0.1), rng.uniform(-math.pi, math.pi)]
        g = [rec[-1, 0] + rng.normal(0, 0.3), rec[-1, 1] + rng.normal(0, 0.3), rng.uniform(-math.pi, math.pi)]
        ops(4, rec, s + g + [int(rng.integers(2, 6))])
        ops(5, rec, [rng.uniform(rec[:, 0].min(), rec[:, 0].max()), rng.normal(0, 1), int(rng.integers(0, n))])
        ops(6, rec, [int(rng.integers(0, n - 1))])
        ops(7, rec, [rng.uniform(0.2, 8), [-1.0, 0.0, 0.5][rng.integers(3)], int(rng.integers(0, 4))])


def test_auto_resize(ops):
    rng = np.random.default_rng(4)
    for _ in range(150):
        n = int(rng.integers(3, 50))
        rec = _band(rng, n)
        dt_ref = rng.uniform(0.1, 0.5)
        ops(11, rec, [dt_ref, dt_ref * rng.uniform(0.05, 0.4), int(rng.integers(3, 6)), int(rng.integers(20, 200)), int(rng.integers(2))])


def test_velocity_command_profile_and_full_trajectory(ops):
    rng = np.random.default_rng(5)
    for _ in range(150):
        n = int(rng.integers(2, 40))
        rec = _band(rng, n)
        max_vel_y = 0.0 if rng.random() < 0.5 else 0.3      # non-holonomic / holonomic extractVelocity (optimal_planner.cpp:1108-1152)
        out = ops(8, rec, [int(rng.integers(1, 6)), max_vel_y])
        assert out[0] in (0.0, 1.0)
        vs = [rng.normal(), rng.normal(), rng.normal(), float(rng.integers(2))]
        vg = [rng.normal(), rng.normal(), rng.normal(), float(rng.integers(2))]
        prof = ops(9, rec, [max_vel_y] + vs + vg)
        assert len(prof) == 3 * (n + 1)
        tr = ops(10, rec, [max_vel_y] + vs + vg)
        assert len(tr) == 7 * n


def test_is_trajectory_feasible_queries_the_same_poses(ops):
    """isTrajectoryFeasible (optimal_planner.cpp:1250-1310) with a costmap stand-in that records every footprint query:
    same verdict, same number of queries and bit-identical queried poses (incl. the interpolated ones between poses that
    are far apart or turned against each other), with a look-ahead index and a look-ahead distance"""
    rng = np.random.default_rng(6)
    for _ in range(200):
        n = int(rng.integers(2, 40))
        rec = _band(rng, n, wiggle=1.5)
        nd = int(rng.integers(0, 4))
        discs = []
        for _k in range(nd):
            i = int(rng.integers(0, n))
            discs += [rec[i, 0] + rng.normal(0, 0.3), rec[i, 1] + rng.normal(0, 0.3), rng.uniform(0.02, 0.25)]
        args = [rng.uniform(0.05, 0.4), rng.uniform(0.4, 0.8), int(rng.integers(-1, n + 2)), [0.0, 1.0, 3.0][int(rng.integers(3))],
                rng.uniform(0.1, 0.6), nd] + discs
        out = ops(12, rec, args)
        assert out[0] in (0.0, 1.0) and len(out) == 2 + 3 * int(out[1])


@pytest.mark.parametrize("kind", [0, 1])
def test_plan_cold_warm_and_reinit_flows(ops, kind):
    """TebOptimalPlanner::plan(start, goal) / plan(initial_plan) call sequences with the optimisation switched off: cold
    start, warm start (updateAndPruneTEB with the moved start / goal) and re-initialisation when the goal jumps beyond
    force_reinit_new_goal_dist / _angular (optimal_planner.cpp:233-321): the band after every call is bit equal"""
    rng = np.random.default_rng(7 + kind)
    for _ in range(80):
        ncalls = int(rng.integers(2, 6))
        head = [kind, ncalls, rng.uniform(0.3, 1.5), rng.uniform(0.2, 1.2), rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8), int(rng.integers(3, 8)),
                int(rng.integers(2)), int(rng.integers(2))]
        body = []
        s = np.array([rng.uniform(-2, 0), rng.uniform(-1, 1), rng.uniform(-1, 1)])
        g = np.array([rng.uniform(3, 5), rng.uniform(-1, 1), rng.uniform(-1, 1)])
        for c in range(ncalls):
            s = s + np.array([rng.uniform(0, 0.3), rng.normal(0, 0.05), rng.normal(0, 0.05)])
            jump = rng.random() < 0.3
            g = g + (np.array([rng.normal(0, 1.5), rng.normal(0, 1.5), rng.normal(0, 1.0)]) if jump else np.array([rng.normal(0, 0.05)] * 3))
            if kind == 0:
                body += s.tolist() + g.tolist()
            else:
                npts = int(rng.integers(2, 12))
                xs = np.linspace(s[0], g[0], npts)
                ys = np.linspace(s[1], g[1], npts) + np.concatenate([[0], rng.normal(0, 0.1, npts - 2), [0]]) if npts > 2 else np.linspace(s[1], g[1], npts)
                th = np.linspace(s[2], g[2], npts)
                body += [npts] + np.stack([xs, ys, th], 1).reshape(-1).tolist()
        out = ops(13, None, head + body)
        assert len(out) > ncalls
