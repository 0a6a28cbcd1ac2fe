"""ctypes binding of oracle/_ref/libteb_ref.so — the REFERENCE'S OWN sources (src/optimal_planner.cpp,
src/timed_elastic_band.cpp, src/obstacles.cpp and the headers they include) compiled against the shims in
oracle/ref_shims/ (Eigen / boost / ROS message stand-ins and a restated g2o optimizer). TEST INFRASTRUCTURE: it pins the
oracle restatement; nothing in the product may load it.

The library can only be built next to the reference's sources (`make -C oracle ref`). The tests that pin against it
read the reference's results from tests/golden/golden_pin_v1.npz through `Pins`; tests/golden/make_golden_pin.py
records that file by running the same tests against the library."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

from teb_local_planner_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libteb_ref.so")
REFERENCE_TREE = "/root/reference"
GOLDEN_PIN = os.path.join(ROOT, "tests", "golden", "golden_pin_v1.npz")
RECORD = None       # {key: Pins} while make_golden_pin.py records GOLDEN_PIN from the library

_lib = None
_golden = None


def _leaves(x):
    """a result as a flat list of float64 arrays: tuples / lists in order, complex as (re, im), -0.0 as 0.0"""
    if isinstance(x, (tuple, list)):
        return [a for y in x for a in _leaves(y)]
    if isinstance(x, complex):
        x = (x.real, x.imag)
    return [np.asarray(x, dtype=np.float64) + 0.0]


def digest(x):
    """128-bit digest of a result's shapes and float64 bits (equal digests <=> np.array_equal on every leaf, for
    results without NaN)"""
    h = hashlib.sha256()
    for a in _leaves(x):
        h.update(np.array(a.shape, np.int64).tobytes())
        h.update(np.ascontiguousarray(a).tobytes())
    return h.digest()[:16]


class Pins:
    """The reference's results one test compares against, in call order. Bit-equality checks keep a digest of the
    reference's result (the results of some tests run to hundreds of MB); tolerance checks keep the values, in float64
    or, where the test allows for the rounding, float32."""
    STREAMS = {np.dtype(np.float64): "/values", np.dtype(np.float32): "/values32"}

    def __init__(self, key):
        self.key, self.nd, self.nl = key, 0, 0
        self.nv = dict.fromkeys(self.STREAMS.values(), 0)
        if RECORD is not None:
            self.digests, self.layout = [], []
            self.values = {s: [] for s in self.STREAMS.values()}
            RECORD[key] = self
            return
        global _golden
        if _golden is None:
            _golden = np.load(GOLDEN_PIN, allow_pickle=False)
        get = lambda s: _golden[key + s] if key + s in _golden.files else np.zeros(0)
        self.digests, self.layout = get("/digests"), get("/layout")
        self.values = {s: get(s) for s in self.STREAMS.values()}

    def equal(self, live, mine, what=""):
        """assert that `mine` is bit equal to the reference's result `live()`"""
        got = digest(mine)
        if RECORD is not None:
            self.digests.append(digest(live()))
        assert self.nd < len(self.digests), f"{self.key}: no stored reference result #{self.nd} (make_golden_pin.py)"
        want = bytes(self.digests[self.nd])
        self.nd += 1
        assert got == want, f"{self.key} #{self.nd - 1} {what}: differs from the reference's result"

    def value(self, live, dtype=np.float64):
        """the reference's result `live()` as a list of float64 arrays (see _leaves), stored as `dtype`"""
        stream = self.STREAMS[np.dtype(dtype)]
        if RECORD is not None:
            leaves = [a.astype(dtype).astype(np.float64) for a in _leaves(live())]
            self.layout += [len(leaves)] + [k for a in leaves for k in (a.ndim, *a.shape)]
            self.values[stream] += [a.reshape(-1).astype(dtype) for a in leaves]
            return leaves
        assert self.nl < len(self.layout), f"{self.key}: no stored reference result (make_golden_pin.py)"
        out, L = [], self.layout
        count, self.nl = int(L[self.nl]), self.nl + 1
        for _ in range(count):
            nd = int(L[self.nl])
            shape = tuple(int(s) for s in L[self.nl + 1:self.nl + 1 + nd])
            self.nl += 1 + nd
            size, at = int(np.prod(shape)), self.nv[stream]
            out.append(self.values[stream][at:at + size].astype(np.float64).reshape(shape))
            self.nv[stream] += size
        return out

    def arrays(self):
        """what GOLDEN_PIN stores for this test"""
        out = {}
        if self.digests:
            out[self.key + "/digests"] = np.frombuffer(b"".join(self.digests), np.uint8).reshape(-1, 16)
        if self.layout:
            out[self.key + "/layout"] = np.array(self.layout, np.int64)
        for stream, vals in self.values.items():
            if vals:
                out[self.key + stream] = np.concatenate(vals)
        return out


@pytest.fixture
def pins(request):
    return Pins(f"{request.module.__name__.rsplit('.', 1)[-1]}::{request.node.name}")


def build_ref():
    if os.path.isdir(REFERENCE_TREE):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "-s", "ref"])
    return REF_SO


def available():
    try:
        build_ref()
    except Exception:
        pass
    return os.path.exists(REF_SO)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError("oracle/_ref/libteb_ref.so is missing (it can only be built where /root/reference exists)")
        L = C.CDLL(REF_SO)
        vp, d, i = C.c_void_p, C.c_double, C.c_int32
        L.teb_ref_abi.restype = i
        L.teb_ref_default_params.restype = None
        L.teb_ref_default_params.argtypes = [C.POINTER(abi.TebParams)]
        L.teb_ref_penalty.restype = d
        L.teb_ref_penalty.argtypes = [i, d, d, d, d]
        L.teb_ref_fast_sigmoid.restype = d
        L.teb_ref_fast_sigmoid.argtypes = [d]
        L.teb_ref_distance.restype = d
        L.teb_ref_distance.argtypes = [vp, vp, vp, vp, d]
        L.teb_ref_auto_resize.restype = i
        L.teb_ref_auto_resize.argtypes = [vp, i, i, d, d, i, i, i]
        L.teb_ref_init_trajectory.restype = i
        L.teb_ref_init_trajectory.argtypes = [vp, vp, d, d, i, i, vp, i]
        L.teb_ref_update_and_prune.restype = i
        L.teb_ref_update_and_prune.argtypes = [vp, i, i, vp, vp, i]
        L.teb_ref_optimize.restype = i
        L.teb_ref_optimize.argtypes = [vp, vp, C.POINTER(i), i, vp, i, vp, vp, i, vp, vp, i, vp, C.POINTER(d), vp]
        L.teb_ref_compute_cost.restype = d
        L.teb_ref_compute_cost.argtypes = [vp, vp, i, vp, i, vp, vp, i, vp, vp, i, vp]
        L.teb_ref_build_system.restype = i
        L.teb_ref_build_system.argtypes = [vp, vp, i, vp, i, vp, vp, i, vp, vp, i, d, vp, vp, C.POINTER(d), vp, i, C.POINTER(i)]
        L.teb_ref_optimize_batch.restype = i
        L.teb_ref_optimize_batch.argtypes = [vp, vp, vp, i, i]
        L.teb_ref_h_signature.restype = i
        L.teb_ref_h_signature.argtypes = [vp, vp, i, vp, i, vp, i, vp, vp]
        L.teb_ref_hcp_explore.restype = i
        L.teb_ref_hcp_explore.argtypes = [vp, vp, vp, vp, vp, i, vp, i, vp, i, vp, i]
        L.teb_ref_hcp_plan.restype = i
        L.teb_ref_hcp_plan.argtypes = [vp, vp, vp, vp, vp, i, vp, i, vp, i, vp, i]
        assert L.teb_ref_abi() == 6
        _lib = L
    return _lib


def _common(obstacles, via, vel_start, vel_goal, obst_vertices):
    ob = np.ascontiguousarray(obstacles, dtype=abi.OBST_DTYPE)
    v = np.zeros((0, 2)) if via is None else np.ascontiguousarray(via, dtype=np.float64).reshape(-1, 2)
    vs = np.array([0, 0, 0, 1.0]) if vel_start is None else np.ascontiguousarray(vel_start, dtype=np.float64)
    vg = np.array([0, 0, 0, 1.0]) if vel_goal is None else np.ascontiguousarray(vel_goal, dtype=np.float64)
    pv = None if obst_vertices is None or len(obst_vertices) == 0 else np.ascontiguousarray(obst_vertices, dtype=np.float64).reshape(-1, 2)
    return ob, v, vs, vg, pv


def default_params():
    p = abi.TebParams()
    lib().teb_ref_default_params(C.byref(p))
    return p


def penalty(which, var, a, b=0.0, eps=0.0):
    return lib().teb_ref_penalty(int(which), float(var), float(a), float(b), float(eps))


def distance(params, pose, obstacle, obst_vertices=None, t=None):
    """calculateDistance (t is None) / estimateSpatioTemporalDistance of the configured footprint to one obstacle"""
    pose = np.ascontiguousarray(pose, dtype=np.float64)
    ob = np.ascontiguousarray(obstacle, dtype=abi.OBST_DTYPE).reshape(1)
    pv = None if obst_vertices is None else np.ascontiguousarray(obst_vertices, dtype=np.float64).reshape(-1, 2)
    return lib().teb_ref_distance(C.addressof(params), pose.ctypes.data, ob.ctypes.data, pv.ctypes.data if pv is not None else None,
                                  -1.0 if t is None else float(t))


def auto_resize(rec, n, dt_ref, dt_hyst, min_samples, max_samples, fast_mode, n_cap=None):
    n_cap = max(rec.shape[0], 4 * n) if n_cap is None else n_cap
    buf = np.zeros((n_cap, 4))
    buf[:n] = rec[:n]
    nn = lib().teb_ref_auto_resize(buf.ctypes.data, n, n_cap, dt_ref, dt_hyst, min_samples, max_samples, int(fast_mode))
    if nn < 0:
        raise RuntimeError("teb_ref_auto_resize: capacity")
    return buf[:nn].copy()


def init_trajectory(start, goal, diststep, max_vel_x, min_samples, backwards=False, n_cap=256):
    buf = np.zeros((n_cap, 4))
    s, g = np.ascontiguousarray(start, dtype=np.float64), np.ascontiguousarray(goal, dtype=np.float64)
    n = lib().teb_ref_init_trajectory(s.ctypes.data, g.ctypes.data, diststep, max_vel_x, min_samples, int(backwards), buf.ctypes.data, n_cap)
    if n < 0:
        raise RuntimeError("teb_ref_init_trajectory: capacity")
    return buf[:n].copy()


def update_and_prune(rec, n, new_start, new_goal, min_samples=3):
    buf = np.ascontiguousarray(rec[:n], dtype=np.float64).copy()
    s, g = np.ascontiguousarray(new_start, dtype=np.float64), np.ascontiguousarray(new_goal, dtype=np.float64)
    nn = lib().teb_ref_update_and_prune(buf.ctypes.data, n, n, s.ctypes.data, g.ctypes.data, min_samples)
    return buf[:nn].copy()


def optimize_band(params, rec, n, obstacles, via=None, vel_start=None, vel_goal=None, rotdir=0, args=None, n_cap=None,
                  obst_vertices=None):
    """TebOptimalPlanner::optimizeTEB of the reference on one band. Returns (rec[n_new], cost, stats dict, ok)."""
    n_cap = rec.shape[0] if n_cap is None else n_cap
    buf = np.zeros((n_cap, 4))
    buf[:n] = rec[:n]
    ob, v, vs, vg, pv = _common(obstacles, via, vel_start, vel_goal, obst_vertices)
    args = abi.make_args(params.no_inner_iterations, params.no_outer_iterations) if args is None else args
    nn = C.c_int32(n)
    cost = C.c_double(np.inf)
    st = np.zeros(6)
    rc = lib().teb_ref_optimize(C.addressof(params), buf.ctypes.data, C.byref(nn), n_cap, ob.ctypes.data if len(ob) else None, len(ob),
                                pv.ctypes.data if pv is not None else None, v.ctypes.data if len(v) else None, len(v),
                                vs.ctypes.data, vg.ctypes.data, int(rotdir), C.addressof(args), C.byref(cost), st.ctypes.data)
    if rc < 0:
        raise RuntimeError("teb_ref_optimize: capacity")
    stats = {"lm_trials": int(st[0]), "rejected": int(st[1]), "terminated": bool(st[2]), "chol_failed": bool(st[3]),
             "diverged": bool(st[4]), "optimized": bool(st[5])}
    return buf[:nn.value].copy(), cost.value, stats, bool(rc)


def optimize_batch(params, hb, args, threads=1, pin=False):
    """In-place on the HostBatch arrays: one band at a time per host thread (the reference's optimizeAllTEBs model)."""
    bs = hb.struct()
    rc = lib().teb_ref_optimize_batch(C.addressof(params), C.addressof(bs), C.addressof(args), int(threads), int(bool(pin)))
    if rc != 0:
        raise RuntimeError(f"teb_ref_optimize_batch rc={rc}")
    return hb


def compute_cost(params, rec, n, obstacles, via=None, vel_start=None, vel_goal=None, rotdir=0, args=None, obst_vertices=None):
    rec = np.ascontiguousarray(rec[:n], dtype=np.float64)
    ob, v, vs, vg, pv = _common(obstacles, via, vel_start, vel_goal, obst_vertices)
    args = abi.make_args() if args is None else args
    return lib().teb_ref_compute_cost(C.addressof(params), rec.ctypes.data, n, ob.ctypes.data if len(ob) else None, len(ob),
                                      pv.ctypes.data if pv is not None else None, v.ctypes.data if len(v) else None, len(v),
                                      vs.ctypes.data, vg.ctypes.data, int(rotdir), C.addressof(args))


def build_system(params, rec, n, obstacles, via=None, vel_start=None, vel_goal=None, rotdir=0, weight_multiplier=1.0,
                 obst_vertices=None, want_edges=False):
    """buildGraph + buildSystem of the reference: dense (H, b, chi2) in g2o order (N = 4n - 7) [+ per-edge rows]."""
    N0 = 4 * n - 7
    H = np.zeros((N0, N0))
    b = np.zeros(N0)
    chi2 = C.c_double(0)
    rec = np.ascontiguousarray(rec[:n], dtype=np.float64)
    ob, v, vs, vg, pv = _common(obstacles, via, vel_start, vel_goal, obst_vertices)
    max_edges = 64 * n + 4 * n * max(len(ob), 1) if want_edges else 0
    edges = np.zeros((max_edges, 64)) if want_edges else None
    ne = C.c_int32(0)
    N = lib().teb_ref_build_system(C.addressof(params), rec.ctypes.data, n, ob.ctypes.data if len(ob) else None, len(ob),
                                   pv.ctypes.data if pv is not None else None, v.ctypes.data if len(v) else None, len(v),
                                   vs.ctypes.data, vg.ctypes.data, int(rotdir), float(weight_multiplier), H.ctypes.data,
                                   b.ctypes.data, C.byref(chi2), edges.ctypes.data if want_edges else None, max_edges, C.byref(ne))
    if N != N0:
        raise RuntimeError(f"teb_ref_build_system: N = {N}, expected {N0}")
    if want_edges:
        return H, b, chi2.value, edges[:ne.value]
    return H, b, chi2.value


def h_signature(params, rec, n, obstacles, use_timediffs=True, obst_vertices=None):
    """calculateEquivalenceClass by the reference's own h_signature.h: complex H (2-D) or M values (x-y-t), plus
    (isValid, isReasonable)"""
    rec = np.ascontiguousarray(rec[:n], dtype=np.float64)
    ob = np.ascontiguousarray(obstacles, dtype=abi.OBST_DTYPE)
    pv = None if obst_vertices is None or len(obst_vertices) == 0 else np.ascontiguousarray(obst_vertices, dtype=np.float64).reshape(-1, 2)
    out = np.zeros(max(2, len(ob)))
    flags = np.zeros(2, np.int32)
    rc = lib().teb_ref_h_signature(C.addressof(params), rec.ctypes.data, n, ob.ctypes.data if len(ob) else None, len(ob),
                                   pv.ctypes.data if pv is not None else None, int(use_timediffs), out.ctypes.data, flags.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"teb_ref_h_signature rc={rc}")
    val = out[:len(ob)].copy() if params.include_dynamic_obstacles else complex(out[0], out[1])
    return val, bool(flags[0]), bool(flags[1])


def hcp_explore(params, hcp, start, goal, obstacles, obst_vertices=None, cycles=1, prm=False):
    """exploreEquivalenceClassesAndInitTebs of the reference's HomotopyClassPlanner on a fresh planner (clearPlanner()
    between cycles). hcp: dict with max_number_classes, obstacle_heading_threshold and, for the roadmap, area width /
    length scale / number of samples. Returns a list (per cycle) of lists of candidate bands [n][4]."""
    ob = np.ascontiguousarray(obstacles, dtype=abi.OBST_DTYPE)
    pv = None if obst_vertices is None or len(obst_vertices) == 0 else np.ascontiguousarray(obst_vertices, dtype=np.float64).reshape(-1, 2)
    h = np.array([hcp["max_number_classes"], hcp["obstacle_heading_threshold"], hcp.get("roadmap_graph_area_width", 6.0),
                  hcp.get("roadmap_graph_area_length_scale", 1.0), hcp.get("roadmap_graph_no_samples", 15), 1.0 if prm else 0.0])
    s, g = np.ascontiguousarray(start, dtype=np.float64), np.ascontiguousarray(goal, dtype=np.float64)
    cap, ccap = 1 << 18, 4096
    out = np.zeros(cap)
    counts = np.zeros(ccap, np.int32)
    w = lib().teb_ref_hcp_explore(C.addressof(params), h.ctypes.data, s.ctypes.data, g.ctypes.data, ob.ctypes.data if len(ob) else None, len(ob),
                                  pv.ctypes.data if pv is not None else None, cycles, out.ctypes.data, cap, counts.ctypes.data, ccap)
    if w < 0:
        raise RuntimeError("teb_ref_hcp_explore: capacity")
    res, ci, pos = [], cycles, 0
    for c in range(cycles):
        bands = []
        for _ in range(int(counts[c])):
            n = int(counts[ci]); ci += 1
            bands.append(out[pos:pos + 4 * n].reshape(n, 4).copy())
            pos += 4 * n
        res.append(bands)
    return res


def hcp_plan(params, hcp, starts, goal, obstacles, obst_vertices=None, prm=False):
    """consecutive HomotopyClassPlanner::plan(start_c, goal) calls on one reference planner. Returns per cycle
    (ok, best_index, [(cost, band[n][4]), ...])."""
    ob = np.ascontiguousarray(obstacles, dtype=abi.OBST_DTYPE)
    pv = None if obst_vertices is None or len(obst_vertices) == 0 else np.ascontiguousarray(obst_vertices, dtype=np.float64).reshape(-1, 2)
    h = np.array([hcp["max_number_classes"], hcp["obstacle_heading_threshold"], hcp.get("roadmap_graph_area_width", 6.0),
                  hcp.get("roadmap_graph_area_length_scale", 1.0), hcp.get("roadmap_graph_no_samples", 15), 1.0 if prm else 0.0])
    st = np.ascontiguousarray(starts, dtype=np.float64).reshape(-1, 3)
    g = np.ascontiguousarray(goal, dtype=np.float64)
    cycles = len(st)
    cap, ccap = 1 << 20, 1 << 14
    out = np.zeros(cap)
    counts = np.zeros(ccap, np.int32)
    w = lib().teb_ref_hcp_plan(C.addressof(params), h.ctypes.data, st.ctypes.data, g.ctypes.data, ob.ctypes.data if len(ob) else None, len(ob),
                               pv.ctypes.data if pv is not None else None, cycles, out.ctypes.data, cap, counts.ctypes.data, ccap)
    if w < 0:
        raise RuntimeError("teb_ref_hcp_plan: capacity")
    res, ci, pos = [], 3 * cycles, 0
    for c in range(cycles):
        cands = []
        for _ in range(int(counts[3 * c])):
            n = int(counts[ci]); ci += 1
            cost = float(out[pos]); pos += 1
            cands.append((cost, out[pos:pos + 4 * n].reshape(n, 4).copy()))
            pos += 4 * n
        res.append((bool(counts[3 * c + 2]), int(counts[3 * c + 1]), cands))
    return res
