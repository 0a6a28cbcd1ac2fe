"""teb_local_planner_b200 — B200-native (sm_100a) batched Timed-Elastic-Band optimizer.

Python side: ctypes loader for the in-tree CUDA library (C-ABI in include/teb_b200.h) and a thin
`TebGpu` convenience wrapper used by tests and bench.py. There is no CPU fallback: if the CUDA
library is missing or no GPU is present, loading / creating a context raises.
"""
import ctypes as C
import os

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libteb_b200.so")
_lib = None


def load_library(build_if_missing=False):
    """Load libteb_b200.so (raises if it has not been built: run `python __graft_entry__.py` / build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import build as _b
            _b.build()
        else:
            raise RuntimeError(f"{LIB_PATH} is missing: build the CUDA extension first "
                               "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.tebgpu_default_params.restype = None
    L.tebgpu_default_params.argtypes = [C.POINTER(abi.TebParams)]
    L.tebgpu_sizeof.restype = C.c_int32
    L.tebgpu_sizeof.argtypes = [C.c_int32]
    L.tebgpu_create.restype = C.c_int32
    L.tebgpu_create.argtypes = [C.POINTER(abi.TebGpuLimits), C.c_int32, C.POINTER(vp)]
    L.tebgpu_destroy.restype = C.c_int32
    L.tebgpu_destroy.argtypes = [vp]
    L.tebgpu_last_error_string.restype = C.c_char_p
    L.tebgpu_last_error_string.argtypes = [vp]
    L.tebgpu_set_params.restype = C.c_int32
    L.tebgpu_set_params.argtypes = [vp, C.POINTER(abi.TebParams)]
    L.tebgpu_optimize_batch.restype = C.c_int32
    L.tebgpu_optimize_batch.argtypes = [vp, C.POINTER(abi.TebBatch), C.POINTER(abi.TebOptimizeArgs)]
    L.tebgpu_optimize_batch_device.restype = C.c_int32
    L.tebgpu_optimize_batch_device.argtypes = [vp, C.POINTER(abi.TebBatch), C.POINTER(abi.TebOptimizeArgs), vp]
    L.tebgpu_set_linearize_variant.restype = C.c_int32
    L.tebgpu_set_linearize_variant.argtypes = [vp, C.c_int32]
    L.tebgpu_set_speculation.restype = C.c_int32
    L.tebgpu_set_speculation.argtypes = [vp, C.c_int32]
    L.tebgpu_set_solver.restype = C.c_int32
    L.tebgpu_set_solver.argtypes = [vp, C.c_int32]
    L.tebgpu_synchronize.restype = C.c_int32
    L.tebgpu_synchronize.argtypes = [vp]
    L.tebgpu_last_launch_count.restype = C.c_int64
    L.tebgpu_last_launch_count.argtypes = [vp]
    L.tebgpu_comm_get_unique_id.restype = C.c_int32
    L.tebgpu_comm_get_unique_id.argtypes = [vp]
    L.tebgpu_comm_init.restype = C.c_int32
    L.tebgpu_comm_init.argtypes = [vp, vp, C.c_int32, C.c_int32]
    L.tebgpu_comm_destroy.restype = C.c_int32
    L.tebgpu_comm_destroy.argtypes = [vp]
    L.tebgpu_gather_costs.restype = C.c_int32
    L.tebgpu_gather_costs.argtypes = [vp, vp, C.c_int32, vp, C.c_int32, vp]
    L.tebgpu_optimize_batch_gather.restype = C.c_int32
    L.tebgpu_optimize_batch_gather.argtypes = [vp, C.POINTER(abi.TebBatch), C.POINTER(abi.TebOptimizeArgs), vp]
    L.tebgpu_set_warp_solver.restype = C.c_int32
    L.tebgpu_set_warp_solver.argtypes = [vp, C.c_int32]
    L.tebgpu_set_graph.restype = C.c_int32
    L.tebgpu_set_graph.argtypes = [vp, C.c_int32]
    L.tebgpu_get_info.restype = C.c_int64
    L.tebgpu_get_info.argtypes = [vp, C.c_int32]
    L.tebgpu_set_profiling.restype = C.c_int32
    L.tebgpu_set_profiling.argtypes = [vp, C.c_int32]
    L.tebgpu_get_kernel_times.restype = C.c_int32
    L.tebgpu_get_kernel_times.argtypes = [vp, C.POINTER(C.c_double * 9), C.POINTER(C.c_int64 * 9)]
    L.tebgpu_compute_cost.restype = C.c_int32
    L.tebgpu_compute_cost.argtypes = [vp, C.POINTER(abi.TebBatch), C.POINTER(abi.TebOptimizeArgs)]
    L.tebgpu_h_signature.restype = C.c_int32
    L.tebgpu_h_signature.argtypes = [vp, C.POINTER(abi.TebBatch), C.c_int32, vp, C.c_int32]
    L.tebgpu_build_system.restype = C.c_int32
    L.tebgpu_build_system.argtypes = [vp, C.POINTER(abi.TebBatch), C.c_int32, vp, vp, C.c_int32]
    L.tebgpu_solve_system.restype = C.c_int32
    L.tebgpu_solve_system.argtypes = [vp, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_int32, vp, vp, vp]
    L.tebgpu_select_best.restype = C.c_int32
    L.tebgpu_select_best.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double]
    L.tebgpu_auto_resize_host.restype = C.c_int32
    L.tebgpu_auto_resize_host.argtypes = [vp, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_int32]
    for which, st in enumerate((abi.TebParams, abi.TebObstacle, abi.TebBatch, abi.TebOptimizeArgs, abi.TebGpuLimits)):
        if L.tebgpu_sizeof(which) != C.sizeof(st):
            raise RuntimeError(f"ABI mismatch for {st.__name__}: C {L.tebgpu_sizeof(which)} vs ctypes {C.sizeof(st)}")
    _lib = L
    return L


class TebGpuError(RuntimeError):
    pass


class TebGpu:
    """One tebgpu context (one device, one stream, its workspaces)."""

    def __init__(self, max_bands, max_poses, max_scenes=1, max_obstacles=64, max_viapoints=0, device=0, max_obst_vertices=0):
        self.lib = load_library()
        lim = abi.TebGpuLimits(max_bands, max_poses, max_scenes, max_obstacles, max_viapoints, max_obst_vertices)
        self.ctx = C.c_void_p()
        rc = self.lib.tebgpu_create(C.byref(lim), device, C.byref(self.ctx))
        if rc != 0:
            msg = self.lib.tebgpu_last_error_string(self.ctx).decode() if self.ctx else ""
            if self.ctx:
                self.lib.tebgpu_destroy(self.ctx)
                self.ctx = None
            raise TebGpuError(f"tebgpu_create failed rc={rc} {msg}")

    def _check(self, rc, what):
        if rc != 0:
            raise TebGpuError(f"{what} rc={rc}: {self.lib.tebgpu_last_error_string(self.ctx).decode()}")

    def set_params(self, params):
        self._check(self.lib.tebgpu_set_params(self.ctx, C.byref(params)), "tebgpu_set_params")
        self.params = params

    def optimize(self, hb, args):
        """Host-buffer call: hb is an abi.HostBatch, updated in place."""
        bs = hb.struct()
        self._check(self.lib.tebgpu_optimize_batch(self.ctx, C.byref(bs), C.byref(args)), "tebgpu_optimize_batch")
        return hb

    def compute_cost(self, hb, args):
        bs = hb.struct()
        self._check(self.lib.tebgpu_compute_cost(self.ctx, C.byref(bs), C.byref(args)), "tebgpu_compute_cost")
        return hb

    def optimize_device(self, batch_struct, args, stream=None):
        self._check(self.lib.tebgpu_optimize_batch_device(self.ctx, C.byref(batch_struct), C.byref(args), stream),
                    "tebgpu_optimize_batch_device")

    def set_linearize_variant(self, v):
        self._check(self.lib.tebgpu_set_linearize_variant(self.ctx, int(v)), "tebgpu_set_linearize_variant")

    def set_speculation(self, k):
        self._check(self.lib.tebgpu_set_speculation(self.ctx, int(k)), "tebgpu_set_speculation")

    def set_warp_solver(self, mode):
        """solve kernel mapping: 0 thread per system, 1 warp per system, 2 by regime"""
        self._check(self.lib.tebgpu_set_warp_solver(self.ctx, int(mode)), "tebgpu_set_warp_solver")

    def set_graph(self, mode):
        """CUDA-graph replay of the launch sequence: 0 never, 1 always, 2 automatic (latency regime)"""
        self._check(self.lib.tebgpu_set_graph(self.ctx, int(mode)), "tebgpu_set_graph")

    def set_solver(self, solver):
        self._check(self.lib.tebgpu_set_solver(self.ctx, int(solver)), "tebgpu_set_solver")

    def synchronize(self):
        self._check(self.lib.tebgpu_synchronize(self.ctx), "tebgpu_synchronize")

    def set_profiling(self, enable):
        self._check(self.lib.tebgpu_set_profiling(self.ctx, int(enable)), "tebgpu_set_profiling")

    def kernel_times(self):
        """{kernel name: (total ms, launches)} since profiling was enabled / last read."""
        ms, cnt = (C.c_double * 9)(), (C.c_int64 * 9)()
        self._check(self.lib.tebgpu_get_kernel_times(self.ctx, C.byref(ms), C.byref(cnt)), "tebgpu_get_kernel_times")
        names = ("k_begin", "k_auto_resize", "k_build_graph", "k_linearize", "k_lm_step_or_retry_rounds", "k_finalize",
                 "k_solve_tpb", "k_trial_eval", "unused")
        return {nme: (ms[i], cnt[i]) for i, nme in enumerate(names)}

    def h_signature(self, hb, use_timediffs=True):
        """calculateEquivalenceClass for every band: complex array [B] (2-D) or float array [B][M_cap] (x-y-t)"""
        import numpy as np
        three_d = bool(self.params.include_dynamic_obstacles) if hasattr(self, "params") else False
        out = np.zeros((hb.B, max(hb.M_cap, 1) if three_d else 2))
        bs = hb.struct()
        self._check(self.lib.tebgpu_h_signature(self.ctx, C.byref(bs), int(use_timediffs), out.ctypes.data, 0),
                    "tebgpu_h_signature")
        return out if three_d else out[:, 0] + 1j * out[:, 1]

    # ---- the one collective (NCCL all-gather of the per-candidate costs), behind the C-ABI
    def comm_get_unique_id(self, out128):
        """rank 0: fill the 128-byte numpy uint8 array with a fresh NCCL unique id"""
        rc = self.lib.tebgpu_comm_get_unique_id(out128.ctypes.data)
        if rc != 0:
            raise TebGpuError(f"tebgpu_comm_get_unique_id rc={rc} (NCCL not loadable?)")

    def comm_init(self, ident128, world, rank):
        self._check(self.lib.tebgpu_comm_init(self.ctx, ident128.ctypes.data, int(world), int(rank)), "tebgpu_comm_init")

    def comm_destroy(self):
        self._check(self.lib.tebgpu_comm_destroy(self.ctx), "tebgpu_comm_destroy")

    def gather_costs_device(self, d_local_ptr, count_local, d_all_ptr, stream=None):
        """device pointers, stream ordered on `stream` (cudaStream_t handle; None = the context's stream)"""
        self._check(self.lib.tebgpu_gather_costs(self.ctx, d_local_ptr, int(count_local), d_all_ptr, 1, stream),
                    "tebgpu_gather_costs")

    def gather_costs(self, local_cost):
        """host numpy vector [count] -> [world * count]"""
        import numpy as np
        local_cost = np.ascontiguousarray(local_cost, dtype=np.float64)
        out = np.zeros(self.info(3) * local_cost.size)
        self._check(self.lib.tebgpu_gather_costs(self.ctx, local_cost.ctypes.data, local_cost.size, out.ctypes.data, 0, None),
                    "tebgpu_gather_costs")
        return out

    def optimize_gather(self, hb, args):
        """tebgpu_optimize_batch + all-gather of the costs: returns the gathered [world * B] vector"""
        import numpy as np
        bs = hb.struct()
        out = np.zeros(self.info(3) * hb.B)
        self._check(self.lib.tebgpu_optimize_batch_gather(self.ctx, C.byref(bs), C.byref(args), out.ctypes.data),
                    "tebgpu_optimize_batch_gather")
        return out

    def info(self, which):
        return int(self.lib.tebgpu_get_info(self.ctx, int(which)))

    def speculation_width(self):
        """speculation width (trials solved concurrently per round) chosen by the last optimize call"""
        return self.info(0)

    def launch_count(self):
        return int(self.lib.tebgpu_last_launch_count(self.ctx))

    def build_system(self, hb, outer_index=0):
        """Returns (Hb [B][4*n_cap][12], chi2 [B]) as numpy arrays (host-buffer path)."""
        import numpy as np
        Hb = np.zeros((hb.B, 4 * hb.n_cap, 12))
        chi2 = np.zeros(hb.B)
        bs = hb.struct()
        self._check(self.lib.tebgpu_build_system(self.ctx, C.byref(bs), outer_index, Hb.ctypes.data, chi2.ctypes.data, 0),
                    "tebgpu_build_system")
        return Hb, chi2

    def solve_system(self, Hb, n, lam, ni, K):
        """LM linear solve only, with the mapping chosen by set_warp_solver: Hb [B][4*n_cap][12] (build_system's
        layout), n [B], lam / ni [B] (damping state before trial 0), K trials per band.
        Returns (dx [B][K][4*n_cap], ok [B][K], lam_used [B][K])."""
        import numpy as np
        Hb = np.ascontiguousarray(Hb, dtype=np.float64)
        B, rows = Hb.shape[0], Hb.shape[1]
        if Hb.shape[2] != 12 or rows % 4:
            raise ValueError(f"Hb must be [B][4*n_cap][12], got {Hb.shape}")
        n = np.ascontiguousarray(n, dtype=np.int32)
        lam = np.ascontiguousarray(np.broadcast_to(lam, (B,)), dtype=np.float64)
        ni = np.ascontiguousarray(np.broadcast_to(ni, (B,)), dtype=np.float64)
        dx = np.empty((B, K, rows))
        ok = np.empty((B, K), dtype=np.int32)
        lam_used = np.empty((B, K))
        self._check(self.lib.tebgpu_solve_system(self.ctx, B, rows // 4, n.ctypes.data, Hb.ctypes.data, lam.ctypes.data,
                                                 ni.ctypes.data, int(K), dx.ctypes.data, ok.ctypes.data,
                                                 lam_used.ctypes.data), "tebgpu_solve_system")
        return dx, ok, lam_used

    def close(self):
        if self.ctx:
            self.lib.tebgpu_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
