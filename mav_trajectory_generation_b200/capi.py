"""ctypes binding of the C-ABI (include/mtg_b200.h) for tests, bench.py and smoke().

This is plumbing only: device memory comes from torch tensors (data_ptr), streams from
torch.cuda.  There is NO fallback: if libmtg_b200.so is missing or no sm_100 device is present
every entry point raises.
"""
import ctypes as C
import os

import numpy as np

from . import _build

MTG_OK = 0
KERNEL_WAYPOINT, KERNEL_GENERIC, KERNEL_NOFREE = 1, 2, 3
STATUS_BAD_TIME, STATUS_NOT_SPD = 1, 2
OPT_WAYPOINT_VARIANT = 1
OPT_RING_DEPTH, OPT_CTAS_PER_SM, OPT_STAGGER_US, OPT_DYNAMIC_TILES, OPT_CHUNK_BLOCKS = 2, 3, 4, 5, 6
OPT_GENERIC_VARIANT = 7
OPT_MELLINGER_UNFUSED = 8
OPT_TMA_INPUTS = 9
OPT_EARLY_REFILL = 10
OPT_V5_STATIC_SHAPE = 11

EXPORTED_SYMBOLS = [
    "mtg_create", "mtg_destroy", "mtg_last_error", "mtg_launch_count", "mtg_device_is_sm100",
    "mtg_problem_layout", "mtg_solve_linear_batch_f64", "mtg_coeffs_from_constraints_batch_f64",
    "mtg_compute_cost_batch_f64", "mtg_solve_linear_batch_host_f64",
    "mtg_coeffs_from_constraints_batch_host_f64", "mtg_compute_cost_batch_host_f64",
    "mtg_host_alloc", "mtg_host_free", "mtg_device_alloc", "mtg_device_free", "mtg_memcpy_h2d",
    "mtg_memcpy_d2h", "mtg_stream_synchronize", "mtg_version", "mtg_set_option",
    "mtg_solve_waypoints_nfabian_batch_f64", "mtg_solve_waypoints_nfabian_batch_host_f64",
    "mtg_cost_gradient_mellinger_batch_f64", "mtg_evaluate_batch_f64", "mtg_evaluate_range_batch_f64",
    "mtg_cost_gradient_mellinger_batch_host_f64", "mtg_evaluate_range_batch_host_f64",
    "mtg_memcpy_d2d", "mtg_ipc_export", "mtg_ipc_import", "mtg_ipc_close",
]


class MtgProblem(C.Structure):
    _fields_ = [("N", C.c_int32), ("r", C.c_int32), ("K", C.c_int32), ("D", C.c_int32),
                ("fixed_mask", C.POINTER(C.c_uint8))]


class MtgLayout(C.Structure):
    _fields_ = [("n_all", C.c_int32), ("n_fixed", C.c_int32), ("n_free", C.c_int32), ("kernel", C.c_int32)]


_lib = None


def load():
    """Load libmtg_b200.so (built in-tree by __graft_entry__.build()).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_CUDA
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the CUDA extension is the only compute path; there is no fallback)")
    L = C.CDLL(path)
    vp, i64, dp = C.c_void_p, C.c_int64, C.c_void_p
    L.mtg_create.restype = C.c_int
    L.mtg_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.mtg_destroy.argtypes = [vp]
    L.mtg_destroy.restype = None
    L.mtg_last_error.restype = C.c_char_p
    L.mtg_last_error.argtypes = [vp]
    L.mtg_launch_count.restype = i64
    L.mtg_launch_count.argtypes = [vp]
    L.mtg_device_is_sm100.argtypes = [vp]
    L.mtg_problem_layout.argtypes = [C.POINTER(MtgProblem), C.POINTER(MtgLayout), vp]
    L.mtg_solve_linear_batch_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, dp, dp, vp]
    L.mtg_coeffs_from_constraints_batch_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, dp, vp]
    L.mtg_compute_cost_batch_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, vp]
    L.mtg_solve_linear_batch_host_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, dp, dp]
    L.mtg_coeffs_from_constraints_batch_host_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, dp]
    L.mtg_compute_cost_batch_host_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp]
    L.mtg_host_alloc.restype = vp
    L.mtg_host_alloc.argtypes = [vp, C.c_uint64]
    L.mtg_host_free.argtypes = [vp, vp]
    L.mtg_device_alloc.restype = vp
    L.mtg_device_alloc.argtypes = [vp, C.c_uint64]
    L.mtg_device_free.argtypes = [vp, vp]
    L.mtg_memcpy_h2d.argtypes = [vp, vp, vp, C.c_uint64, vp]
    L.mtg_memcpy_d2h.argtypes = [vp, vp, vp, C.c_uint64, vp]
    L.mtg_stream_synchronize.argtypes = [vp, vp]
    L.mtg_memcpy_d2d.argtypes = [vp, vp, vp, C.c_uint64, vp]
    L.mtg_ipc_export.argtypes = [vp, vp, C.c_char_p, C.POINTER(C.c_uint64)]
    L.mtg_ipc_import.argtypes = [vp, C.c_char_p, C.c_uint64, C.POINTER(vp), C.POINTER(vp)]
    L.mtg_ipc_close.argtypes = [vp, vp]
    L.mtg_version.restype = C.c_int
    L.mtg_set_option.argtypes = [vp, C.c_int, C.c_int]
    L.mtg_evaluate_batch_f64.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, i64, dp, dp, C.c_int32, C.c_double,
                                         C.c_double, C.c_int32, dp, vp]
    L.mtg_evaluate_range_batch_f64.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, i64, dp, dp, C.c_double, C.c_double,
                                               C.c_double, C.c_int32, C.POINTER(C.c_int32), C.c_int32, dp, dp, dp, vp]
    L.mtg_cost_gradient_mellinger_batch_f64.argtypes = [vp, C.POINTER(MtgProblem), i64, dp, dp, dp, dp, vp]
    L.mtg_solve_waypoints_nfabian_batch_host_f64.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, i64, dp,
                                                             C.c_double, C.c_double, C.c_double, dp, dp, dp]
    L.mtg_solve_waypoints_nfabian_batch_f64.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, i64, dp,
                                                        C.c_double, C.c_double, C.c_double, dp, dp, dp, vp]
    for name in EXPORTED_SYMBOLS:
        getattr(L, name)  # AttributeError if the library does not export what the header declares
    _lib = L
    return L


class Problem:
    """A constraint topology: N, derivative_to_optimize r, K segments, D dimensions and the
    per-vertex fixed mask ([K+1][N/2], None = createRandomVertices topology)."""

    def __init__(self, N, r, K, D, fixed_mask=None):
        self.N, self.r, self.K, self.D = int(N), int(r), int(K), int(D)
        self._mask = None
        self.c = MtgProblem(self.N, self.r, self.K, self.D, None)
        if fixed_mask is not None:
            self._mask = np.ascontiguousarray(fixed_mask, dtype=np.uint8).reshape(self.K + 1, self.N // 2)
            self.c.fixed_mask = self._mask.ctypes.data_as(C.POINTER(C.c_uint8))
        lay = MtgLayout()
        slot = np.zeros(max(self.K * self.N, 1), dtype=np.int32)
        rc = load().mtg_problem_layout(C.byref(self.c), C.byref(lay), slot.ctypes.data)
        if rc != MTG_OK:
            raise ValueError(f"invalid problem N={N} r={r} K={K} D={D} (rc={rc})")
        self.n_all, self.n_fixed, self.n_free, self.kernel = lay.n_all, lay.n_fixed, lay.n_free, lay.kernel
        self.slot_col = slot[: self.K * self.N]

    @property
    def bytes_per_trajectory(self):
        """Algorithmic HBM bytes: seg_times + d_fixed in, coeffs out (SURVEY.md 8d)."""
        return 8 * (self.K + self.D * self.n_fixed) + 8 * self.K * self.D * self.N


class Solver:
    """One handle on one CUDA device (single caller)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.mtg_create(int(device), C.byref(h))
        if rc != MTG_OK:
            raise RuntimeError(f"mtg_create failed (rc={rc}): {self.lib.mtg_last_error(None).decode()}")
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.mtg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != MTG_OK:
            raise RuntimeError(f"{what} failed (rc={rc}): {self.lib.mtg_last_error(self.h).decode()}")

    def set_option(self, key, value):
        self._check(self.lib.mtg_set_option(self.h, int(key), int(value)), "mtg_set_option")

    @property
    def launch_count(self):
        return int(self.lib.mtg_launch_count(self.h))

    # ---- device-pointer path (torch CUDA tensors, float64, contiguous) --------------------
    def solve_linear(self, prob, seg_times, d_fixed, coeffs=None, d_free=None, status=None, stream=None):
        import torch
        B = seg_times.shape[0]
        assert seg_times.is_cuda and seg_times.dtype == torch.float64 and seg_times.is_contiguous()
        assert d_fixed.is_cuda and d_fixed.dtype == torch.float64 and d_fixed.is_contiguous()
        assert tuple(seg_times.shape) == (B, prob.K) and tuple(d_fixed.shape) == (B, prob.D, prob.n_fixed)
        if coeffs is None:
            coeffs = torch.empty((B, prob.K, prob.D, prob.N), dtype=torch.float64, device=seg_times.device)
        assert coeffs.is_contiguous() and tuple(coeffs.shape) == (B, prob.K, prob.D, prob.N)
        s = stream if stream is not None else torch.cuda.current_stream(seg_times.device).cuda_stream
        rc = self.lib.mtg_solve_linear_batch_f64(
            self.h, C.byref(prob.c), B, seg_times.data_ptr(), d_fixed.data_ptr(), coeffs.data_ptr(),
            d_free.data_ptr() if d_free is not None else None,
            status.data_ptr() if status is not None else None, s)
        self._check(rc, "mtg_solve_linear_batch_f64")
        return coeffs

    # ---- raw device pointers (peer memory imported with ipc_import has no torch tensor behind it) ----
    def solve_linear_ptr(self, prob, B, seg_times_ptr, d_fixed_ptr, coeffs_ptr, stream):
        rc = self.lib.mtg_solve_linear_batch_f64(self.h, C.byref(prob.c), int(B), int(seg_times_ptr), int(d_fixed_ptr),
                                                 int(coeffs_ptr), None, None, int(stream))
        self._check(rc, "mtg_solve_linear_batch_f64")

    def memcpy_d2d(self, dst_ptr, src_ptr, nbytes, stream):
        self._check(self.lib.mtg_memcpy_d2d(self.h, int(dst_ptr), int(src_ptr), int(nbytes), int(stream)), "mtg_memcpy_d2d")

    def ipc_export(self, tensor):
        """(handle bytes [64], offset) of a CUDA tensor's storage position, for ipc_import on another rank."""
        buf = C.create_string_buffer(64)
        off = C.c_uint64(0)
        self._check(self.lib.mtg_ipc_export(self.h, tensor.data_ptr(), buf, C.byref(off)), "mtg_ipc_export")
        return bytes(buf.raw), int(off.value)

    def ipc_import(self, handle, offset):
        """-> (pointer to the exported position, base pointer to pass to ipc_close)."""
        ptr, base = C.c_void_p(), C.c_void_p()
        self._check(self.lib.mtg_ipc_import(self.h, handle, int(offset), C.byref(ptr), C.byref(base)), "mtg_ipc_import")
        return int(ptr.value), int(base.value)

    def ipc_close(self, base):
        self._check(self.lib.mtg_ipc_close(self.h, int(base)), "mtg_ipc_close")

    def solve_waypoints_nfabian(self, N, r, positions, v_max, a_max, magic=6.5, coeffs=None, seg_times_out=None,
                                status=None, stream=None):
        """positions: CUDA float64 [B][K+1][D] -> coeffs [B][K][D][N] (fused Nfabian times + packing)."""
        import torch
        B, K1, D = positions.shape
        K = K1 - 1
        assert positions.is_cuda and positions.dtype == torch.float64 and positions.is_contiguous()
        if coeffs is None:
            coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=positions.device)
        s = stream if stream is not None else torch.cuda.current_stream(positions.device).cuda_stream
        rc = self.lib.mtg_solve_waypoints_nfabian_batch_f64(
            self.h, N, r, K, D, B, positions.data_ptr(), float(v_max), float(a_max), float(magic), coeffs.data_ptr(),
            seg_times_out.data_ptr() if seg_times_out is not None else None,
            status.data_ptr() if status is not None else None, s)
        self._check(rc, "mtg_solve_waypoints_nfabian_batch_f64")
        return coeffs

    def evaluate(self, seg_times, coeffs, derivative, t_start, dt, n_samples, stream=None):
        """coeffs [B][K][D][N] -> samples [B][n_samples][D] of the given derivative (Trajectory::evaluate)."""
        import torch
        B, K, D, N = coeffs.shape
        out = torch.empty((B, n_samples, D), dtype=torch.float64, device=coeffs.device)
        s = stream if stream is not None else torch.cuda.current_stream(coeffs.device).cuda_stream
        rc = self.lib.mtg_evaluate_batch_f64(self.h, N, K, D, B, seg_times.data_ptr(), coeffs.data_ptr(),
                                             int(derivative), float(t_start), float(dt), int(n_samples),
                                             out.data_ptr(), s)
        self._check(rc, "mtg_evaluate_batch_f64")
        return out

    def evaluate_range(self, seg_times, coeffs, t_start, t_end, dt, derivs=(0,), max_samples=None, want_times=False,
                       stream=None):
        """Batched Trajectory::evaluateRange: (out [B][S][len(derivs)][D], n_samples [B] int32, sampling_times or None)."""
        import torch
        B, K, D, N = coeffs.shape
        if max_samples is None:
            max_samples = int((t_end - t_start) / dt + 1) + 2
        derivs = [int(x) for x in derivs]
        arr = (C.c_int32 * len(derivs))(*derivs)
        out = torch.empty((B, max_samples, len(derivs), D), dtype=torch.float64, device=coeffs.device)
        n = torch.empty((B,), dtype=torch.int32, device=coeffs.device)
        st = torch.zeros((B, max_samples), dtype=torch.float64, device=coeffs.device) if want_times else None
        s = stream if stream is not None else torch.cuda.current_stream(coeffs.device).cuda_stream
        rc = self.lib.mtg_evaluate_range_batch_f64(self.h, N, K, D, B, seg_times.data_ptr(), coeffs.data_ptr(),
                                                   float(t_start), float(t_end), float(dt), len(derivs), arr,
                                                   int(max_samples), out.data_ptr(), n.data_ptr(),
                                                   st.data_ptr() if want_times else None, s)
        self._check(rc, "mtg_evaluate_range_batch_f64")
        return out, n, st

    def cost_gradient_mellinger(self, prob, seg_times, d_fixed, stream=None):
        """(cost [B], grad [B][K]) -- batched getCostAndGradientMellinger."""
        import torch
        B = seg_times.shape[0]
        cost = torch.empty((B,), dtype=torch.float64, device=seg_times.device)
        grad = torch.empty((B, prob.K), dtype=torch.float64, device=seg_times.device)
        s = stream if stream is not None else torch.cuda.current_stream(seg_times.device).cuda_stream
        rc = self.lib.mtg_cost_gradient_mellinger_batch_f64(self.h, C.byref(prob.c), B, seg_times.data_ptr(),
                                                            d_fixed.data_ptr(), cost.data_ptr(), grad.data_ptr(), s)
        self._check(rc, "mtg_cost_gradient_mellinger_batch_f64")
        return cost, grad

    def coeffs_from_constraints(self, prob, seg_times, d_fixed, d_free, coeffs=None, stream=None):
        import torch
        B = seg_times.shape[0]
        if coeffs is None:
            coeffs = torch.empty((B, prob.K, prob.D, prob.N), dtype=torch.float64, device=seg_times.device)
        s = stream if stream is not None else torch.cuda.current_stream(seg_times.device).cuda_stream
        rc = self.lib.mtg_coeffs_from_constraints_batch_f64(
            self.h, C.byref(prob.c), B, seg_times.data_ptr(), d_fixed.data_ptr(),
            d_free.data_ptr() if d_free is not None else None, coeffs.data_ptr(), s)
        self._check(rc, "mtg_coeffs_from_constraints_batch_f64")
        return coeffs

    def compute_cost(self, prob, seg_times, coeffs, cost=None, stream=None):
        import torch
        B = seg_times.shape[0]
        if cost is None:
            cost = torch.empty((B,), dtype=torch.float64, device=seg_times.device)
        s = stream if stream is not None else torch.cuda.current_stream(seg_times.device).cuda_stream
        rc = self.lib.mtg_compute_cost_batch_f64(self.h, C.byref(prob.c), B, seg_times.data_ptr(),
                                                 coeffs.data_ptr(), cost.data_ptr(), s)
        self._check(rc, "mtg_compute_cost_batch_f64")
        return cost

    # ---- host-pointer path (numpy arrays or pinned torch CPU tensors) ----------------------
    @staticmethod
    def _hptr(a):
        if a is None:
            return None
        if isinstance(a, np.ndarray):
            assert a.flags["C_CONTIGUOUS"]
            return a.ctypes.data
        assert a.is_contiguous() and not a.is_cuda
        return a.data_ptr()

    def solve_linear_host(self, prob, seg_times, d_fixed, coeffs, d_free=None, status=None):
        B = seg_times.shape[0]
        rc = self.lib.mtg_solve_linear_batch_host_f64(
            self.h, C.byref(prob.c), B, self._hptr(seg_times), self._hptr(d_fixed), self._hptr(coeffs),
            self._hptr(d_free), self._hptr(status))
        self._check(rc, "mtg_solve_linear_batch_host_f64")
        return coeffs

    def solve_waypoints_nfabian_host(self, N, r, positions, v_max, a_max, magic, coeffs, seg_times_out=None,
                                     status=None):
        """positions host [B][K+1][D] -> coeffs host [B][K][D][N] (pipelined H2D / fused solve / D2H)."""
        B, K1, D = positions.shape
        rc = self.lib.mtg_solve_waypoints_nfabian_batch_host_f64(
            self.h, N, r, K1 - 1, D, B, self._hptr(positions), float(v_max), float(a_max), float(magic),
            self._hptr(coeffs), self._hptr(seg_times_out), self._hptr(status))
        self._check(rc, "mtg_solve_waypoints_nfabian_batch_host_f64")
        return coeffs

    def coeffs_from_constraints_host(self, prob, seg_times, d_fixed, d_free, coeffs):
        B = seg_times.shape[0]
        rc = self.lib.mtg_coeffs_from_constraints_batch_host_f64(
            self.h, C.byref(prob.c), B, self._hptr(seg_times), self._hptr(d_fixed), self._hptr(d_free),
            self._hptr(coeffs))
        self._check(rc, "mtg_coeffs_from_constraints_batch_host_f64")
        return coeffs

    def compute_cost_host(self, prob, seg_times, coeffs, cost):
        B = seg_times.shape[0]
        rc = self.lib.mtg_compute_cost_batch_host_f64(self.h, C.byref(prob.c), B, self._hptr(seg_times),
                                                      self._hptr(coeffs), self._hptr(cost))
        self._check(rc, "mtg_compute_cost_batch_host_f64")
        return cost
