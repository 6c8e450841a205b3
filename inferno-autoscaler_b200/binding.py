"""ctypes binding of libwva_b200.so (the C-ABI of include/wva_b200.h).

The library holds sm_100a kernels only.  There is no CPU implementation behind this module:
loading fails loudly when the shared object has not been built, and every compute call fails
with WvaError(ECUDA) when no B200 is present.
"""
import ctypes as C
import os

import numpy as np

from . import abi
from .image import SystemImage

_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_DIR, "libwva_b200.so")
_lib = None

# every symbol include/wva_b200.h declares (tests/test_abi_symbols.py checks the header against this)
EXPORTS = [
    "wva_abi_version", "wva_ctx_create", "wva_ctx_destroy", "wva_last_error", "wva_system_upload", "wva_set_shard",
    "wva_analyze_pairs", "wva_pairs_device", "wva_pairs_commit", "wva_pair_steps", "wva_pair_counters", "wva_pair_debug", "wva_analyze_grid",
    "wva_analyze_grid_device", "wva_grid_fetch", "wva_solve", "wva_allocate_by_type", "wva_type_totals_device",
    "wva_solution_time_usec", "wva_queue_analyze", "wva_queue_size", "wva_launch_count", "wva_phase_time_usec",
    "wva_grid_counters", "wva_selftest_division", "wva_stream", "wva_grid_set_tail_cap", "wva_grid_list_sizes", "wva_grid_set_fused", "wva_grid_last_fused", "wva_pairs_set_warp_max", "wva_pairs_set_pstore", "wva_solve_set_ranked", "wva_solve_greedy_path", "wva_solve_stats", "wva_type_totals_merge", "wva_set_certified_tails", "wva_analyze", "wva_pairs_fetch", "wva_grid_deferred_fetch",
    "wva_system_upload_arrays", "wva_analyze_pairs_arrays", "wva_pairs_fetch_arrays", "wva_solve_arrays",
    "wva_system_update_servers", "wva_system_update_models", "wva_system_remove_server", "wva_system_set_capacity", "wva_upload_bytes", "wva_system_dims",
    "wva_model_solve",
    "wva_comm_unique_id", "wva_comm_init", "wva_comm_destroy", "wva_comm_info", "wva_comm_shard",
    "wva_group_create", "wva_group_destroy", "wva_group_size", "wva_group_ctx", "wva_group_last_error", "wva_group_upload",
    "wva_group_analyze", "wva_group_pairs_fetch", "wva_group_grid_fetch", "wva_group_solve", "wva_group_allocate_by_type",
    "wva_grid_set_pair_winners", "wva_grid_pairs_fetch", "wva_grid_pairs_fetch_arrays", "wva_solve_grid", "wva_solve_grid_arrays",
    "wva_group_grid_pairs_fetch", "wva_group_solve_grid",
    "wva_grid_pairs_size", "wva_group_grid_pairs_size",
    "wva_analyze_scenarios", "wva_scenario_pairs_fetch", "wva_analyze_scenarios_arrays", "wva_scenario_pairs_fetch_arrays",
    "wva_group_analyze_scenarios", "wva_group_scenario_pairs_fetch",
]


class WvaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("wva_b200 error %d: %s" % (code, msg))
        self.code = code


def lib():
    """Load libwva_b200.so (built by __graft_entry__.build()).  No fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("CUDA library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU implementation to fall back to)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
        L.wva_abi_version.restype = C.c_int
        L.wva_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.wva_ctx_destroy.argtypes = [vp]
        L.wva_ctx_destroy.restype = None
        L.wva_last_error.argtypes = [vp]
        L.wva_last_error.restype = C.c_char_p
        L.wva_system_upload.argtypes = [vp, C.POINTER(abi.SystemSoa)]
        L.wva_set_shard.argtypes = [vp, i32, i32]
        L.wva_analyze_pairs.argtypes = [vp, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_pairs_device.argtypes = [vp, C.POINTER(abi.AllocSoa), C.POINTER(vp)]
        L.wva_pairs_commit.argtypes = [vp]
        L.wva_pair_steps.argtypes = [vp, C.POINTER(u64)]
        L.wva_pair_counters.argtypes = [vp, C.POINTER(u64)]
        L.wva_pair_debug.argtypes = [vp, C.POINTER(u64), i32]
        L.wva_analyze_grid.argtypes = [vp, i32, i32, vp, vp, vp]
        L.wva_analyze_grid_device.argtypes = [vp, i32, i32, i32]
        L.wva_grid_fetch.argtypes = [vp, vp]
        L.wva_solve.argtypes = [vp, C.POINTER(abi.OptimizerSpec), abi.i32p, C.POINTER(abi.AllocSoa)]
        L.wva_allocate_by_type.argtypes = [vp, abi.i64p, abi.f32p]
        L.wva_type_totals_device.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]
        L.wva_solution_time_usec.argtypes = [vp]
        L.wva_solution_time_usec.restype = i64
        L.wva_queue_analyze.argtypes = [vp, i32, vp, abi.f32p, vp, abi.u8p]
        L.wva_queue_size.argtypes = [vp, i32, vp, abi.f32p, abi.f32p, vp, abi.f32p, abi.u8p]
        L.wva_launch_count.argtypes = [vp]
        L.wva_launch_count.restype = i64
        L.wva_phase_time_usec.argtypes = [vp, C.c_int]
        L.wva_phase_time_usec.restype = i64
        L.wva_grid_counters.argtypes = [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]
        L.wva_selftest_division.argtypes = [vp, u64, u64, C.c_int, C.POINTER(u64)]
        L.wva_pairs_set_warp_max.argtypes = [vp, i32]
        L.wva_pairs_set_pstore.argtypes = [vp, i32]
        L.wva_solve_set_ranked.argtypes = [vp, i32]
        L.wva_solve_greedy_path.argtypes = [vp]
        L.wva_solve_stats.argtypes = [vp, C.POINTER(C.c_uint64)]
        L.wva_type_totals_merge.argtypes = [vp, C.c_void_p, i32]
        L.wva_set_certified_tails.argtypes = [vp, i32]
        L.wva_analyze.argtypes = [vp, i32, i32, i32]
        L.wva_pairs_fetch.argtypes = [vp, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_grid_set_tail_cap.argtypes = [vp, i32]
        L.wva_grid_list_sizes.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
        L.wva_grid_set_fused.argtypes = [vp, i32]
        L.wva_grid_last_fused.argtypes = [vp]
        L.wva_grid_deferred_fetch.argtypes = [vp, C.POINTER(u64), i32, C.POINTER(i32)]
        L.wva_stream.argtypes = [vp]
        L.wva_stream.restype = vp
        L.wva_system_update_servers.argtypes = [vp, i32, i32, C.POINTER(abi.SystemSoa)]
        L.wva_system_update_models.argtypes = [vp, i32, i32, C.POINTER(abi.SystemSoa)]
        L.wva_system_remove_server.argtypes = [vp, i32]
        L.wva_system_set_capacity.argtypes = [vp, abi.i64p]
        L.wva_upload_bytes.argtypes = [vp]
        L.wva_upload_bytes.restype = i64
        L.wva_system_dims.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
        L.wva_model_solve.argtypes = [vp, i64, abi.f32p, i32, i32, abi.f32p, abi.f32p, abi.f32p, C.POINTER(C.c_double)]
        L.wva_comm_unique_id.argtypes = [vp]
        L.wva_comm_init.argtypes = [vp, vp, i32, i32]
        L.wva_comm_destroy.argtypes = [vp]
        L.wva_comm_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
        L.wva_comm_shard.argtypes = [vp]
        L.wva_group_create.argtypes = [abi.i32p, i32, C.POINTER(vp)]
        L.wva_group_destroy.argtypes = [vp]
        L.wva_group_destroy.restype = None
        L.wva_group_size.argtypes = [vp]
        L.wva_group_ctx.argtypes = [vp, i32]
        L.wva_group_ctx.restype = vp
        L.wva_group_last_error.argtypes = [vp]
        L.wva_group_last_error.restype = C.c_char_p
        L.wva_group_upload.argtypes = [vp, C.POINTER(abi.SystemSoa)]
        L.wva_group_analyze.argtypes = [vp, i32, i32, i32]
        L.wva_group_pairs_fetch.argtypes = [vp, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_group_grid_fetch.argtypes = [vp, vp]
        L.wva_group_solve.argtypes = [vp, C.POINTER(abi.OptimizerSpec), abi.i32p, C.POINTER(abi.AllocSoa)]
        L.wva_group_allocate_by_type.argtypes = [vp, abi.i64p, abi.f32p]
        L.wva_grid_set_pair_winners.argtypes = [vp, i32]
        L.wva_grid_pairs_fetch.argtypes = [vp, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_solve_grid.argtypes = [vp, C.POINTER(abi.OptimizerSpec), abi.i32p, C.POINTER(abi.AllocSoa)]
        L.wva_group_grid_pairs_fetch.argtypes = [vp, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_group_solve_grid.argtypes = [vp, C.POINTER(abi.OptimizerSpec), abi.i32p, C.POINTER(abi.AllocSoa)]
        L.wva_grid_pairs_size.argtypes = [vp, abi.u8p]
        L.wva_group_grid_pairs_size.argtypes = [vp, abi.u8p]
        L.wva_analyze_scenarios.argtypes = [vp, i32, abi.f32p, abi.i32p, C.POINTER(abi.AllocSoa), abi.i64p, abi.f32p]
        L.wva_scenario_pairs_fetch.argtypes = [vp, i32, C.POINTER(abi.AllocSoa), abi.u8p]
        L.wva_group_analyze_scenarios.argtypes = [vp, i32, abi.f32p, abi.i32p, C.POINTER(abi.AllocSoa), abi.i64p, abi.f32p]
        L.wva_group_scenario_pairs_fetch.argtypes = [vp, i32, C.POINTER(abi.AllocSoa), abi.u8p]
        if L.wva_abi_version() != abi.ABI_VERSION:
            raise ImportError("libwva_b200.so ABI version mismatch")
        _lib = L
    return _lib


def _status_buffer(status, n):
    """a caller's uint8[n] status buffer (written in place), or a new zeroed one"""
    if status is None:
        return np.zeros(n, dtype=np.uint8)
    if not isinstance(status, np.ndarray) or status.dtype != np.uint8 or status.shape != (n,) or not status.flags.c_contiguous:
        raise ValueError("status must be a contiguous uint8 array of S*A = %d entries" % n)
    return status


def _scenario_rates(arrival_rpm, S):
    """the caller's [L, S] float32 scenario rates, checked before they reach the library"""
    if not isinstance(arrival_rpm, np.ndarray) or arrival_rpm.dtype != np.float32:
        raise TypeError("arrival_rpm must be a float32 numpy array of shape (n_scen, S)")
    if arrival_rpm.ndim != 2 or arrival_rpm.shape[1] != S or not 1 <= arrival_rpm.shape[0] <= abi.MAX_SCENARIOS:
        raise ValueError("arrival_rpm must have shape (n_scen, %d) with 1 <= n_scen <= %d, got %s"
                         % (S, abi.MAX_SCENARIOS, arrival_rpm.shape))
    if not np.isfinite(arrival_rpm).all():
        raise ValueError("arrival_rpm holds NaN or Inf")
    return np.ascontiguousarray(arrival_rpm)


def _analyze_scenarios(fn, h, T, rates):
    L, S = rates.shape
    chosen_acc = np.full(L * S, -1, dtype=np.int32)
    chosen = abi.AllocArrays(L * S)
    count = np.zeros(L * T, dtype=np.int64)
    cost = np.zeros(L * T, dtype=np.float32)
    rc = fn(h, L, abi.ptr(rates, C.c_float), abi.ptr(chosen_acc, C.c_int32), C.byref(chosen.c), abi.ptr(count, C.c_int64),
            abi.ptr(cost, C.c_float))
    return rc, (chosen_acc.reshape(L, S), chosen, count.reshape(L, T), cost.reshape(L, T))


def comm_unique_id():
    """128-byte NCCL id (rank 0 creates it, the host distributes it, every rank passes it to Context.comm_init)."""
    buf = C.create_string_buffer(abi.COMM_ID_BYTES)
    rc = lib().wva_comm_unique_id(buf)
    if rc != abi.OK:
        raise WvaError(rc, lib().wva_last_error(None).decode())
    return bytes(buf.raw)


class Context:
    """wva_ctx: one CUDA device, one stream, one call in flight."""

    def __init__(self, device=0, _borrowed=None):
        self._h = C.c_void_p()
        self._owned = _borrowed is None
        if _borrowed is not None:
            self._h = C.c_void_p(_borrowed)
        else:
            rc = lib().wva_ctx_create(int(device), C.byref(self._h))
            if rc != abi.OK:
                raise WvaError(rc, lib().wva_last_error(None).decode())
        self.device = int(device)
        self.image = None

    def close(self):
        if self._h and self._owned:
            lib().wva_ctx_destroy(self._h)
        self._h = C.c_void_p()

    # ---- multi-rank (one process per GPU) ------------------------------------------------
    def comm_init(self, unique_id, rank, n_ranks):
        assert len(unique_id) == abi.COMM_ID_BYTES
        self._ck(lib().wva_comm_init(self._h, C.c_char_p(unique_id), int(rank), int(n_ranks)))

    def comm_destroy(self):
        self._ck(lib().wva_comm_destroy(self._h))

    def comm_info(self):
        r, n = C.c_int32(0), C.c_int32(1)
        self._ck(lib().wva_comm_info(self._h, C.byref(r), C.byref(n)))
        return r.value, n.value

    def comm_shard(self):
        """this rank's contiguous server range of the uploaded image: floor(S*g/G) boundaries"""
        self._ck(lib().wva_comm_shard(self._h))
        r, n = self.comm_info()
        S = self.image.S
        self.first = S * r // n
        self.count = S * (r + 1) // n - self.first

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != abi.OK:
            raise WvaError(rc, lib().wva_last_error(self._h).decode())

    # ---- system ------------------------------------------------------------------------
    def upload(self, image: SystemImage):
        s = image.c_struct()
        self._ck(lib().wva_system_upload(self._h, C.byref(s)))
        self.image = image
        self.first, self.count = 0, image.S

    # ---- incremental updates of the resident image (system.go:99-171) ------------------------
    def update_servers(self, first, rows: SystemImage):
        """overwrite / append server rows [first, first+rows.S) from `rows` (its server arrays); self.image follows"""
        s = rows.c_struct()
        self._ck(lib().wva_system_update_servers(self._h, int(first), rows.S, C.byref(s)))
        img = self.image
        newS = max(img.S, first + rows.S)
        for name, dt in abi.SRV_FIELDS:
            arr = getattr(img, name)
            if newS > img.S:
                arr = np.concatenate([arr, np.zeros(newS - img.S, dtype=dt)])
            arr[first:first + rows.S] = getattr(rows, name)
            setattr(img, name, arr)
        img.S = newS
        self.first, self.count = 0, newS

    def update_models(self, first, rows: SystemImage):
        s = rows.c_struct()
        self._ck(lib().wva_system_update_models(self._h, int(first), rows.M, C.byref(s)))
        img = self.image
        newM = max(img.M, first + rows.M)
        for name, dt in abi.PERF_FIELDS:
            arr = getattr(img, name)
            if newM > img.M:
                arr = np.concatenate([arr, np.zeros((newM - img.M) * img.A, dtype=dt)])
            arr[first * img.A:(first + rows.M) * img.A] = getattr(rows, name)
            setattr(img, name, arr)
        img.M = newM
        self.first, self.count = 0, img.S

    def remove_server(self, index):
        """RemoveServer: the last server's row moves into `index`; self.image follows"""
        self._ck(lib().wva_system_remove_server(self._h, int(index)))
        img = self.image
        for name, _ in abi.SRV_FIELDS:
            arr = getattr(img, name)
            arr[index] = arr[img.S - 1]
            setattr(img, name, arr[:img.S - 1].copy())
        img.S -= 1
        self.first, self.count = 0, img.S

    def set_capacity(self, type_capacity):
        cap = np.ascontiguousarray(type_capacity, dtype=np.int64)
        self._ck(lib().wva_system_set_capacity(self._h, abi.ptr(cap, C.c_int64)))
        self.image.type_capacity = cap.copy()

    def upload_bytes(self):
        return int(lib().wva_upload_bytes(self._h))

    def dims(self):
        v = [C.c_int32(0) for _ in range(4)]
        self._ck(lib().wva_system_dims(self._h, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)

    def set_shard(self, first, count):
        self._ck(lib().wva_set_shard(self._h, int(first), int(count)))
        self.first, self.count = int(first), int(count)

    # ---- analyze -----------------------------------------------------------------------
    def analyze_pairs(self, download=True):
        """Server.Calculate for the shard.  Returns (AllocArrays[S*A], feasible[S*A]) (rows outside the
        shard are zero) or None when download is False (results stay on the device)."""
        if not download:
            self._ck(lib().wva_analyze_pairs(self._h, None, None))
            return None
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_analyze_pairs(self._h, C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def analyze(self, r_max, b_max, want_cube=False):
        """Server.Calculate for every pair and the candidate sweep, overlapped; results stay on the device."""
        self._ck(lib().wva_analyze(self._h, int(r_max), int(b_max), 1 if want_cube else 0))

    def pairs_fetch(self):
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_pairs_fetch(self._h, C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def pair_counters(self):
        v = (C.c_uint64 * 4)()
        self._ck(lib().wva_pair_counters(self._h, v))
        return dict(steps=v[0], rounds_sum=v[1], rounds_max=v[2], trailing=v[3])

    def set_certified_tails(self, on):
        self._ck(lib().wva_set_certified_tails(self._h, int(on)))

    def pair_debug(self):
        n = self.count * self.image.A
        out = np.zeros(2 * n, dtype=np.uint64)
        self._ck(lib().wva_pair_debug(self._h, out.ctypes.data_as(C.POINTER(C.c_uint64)), n))
        return out.reshape(n, 2)

    def pairs_set_pstore(self, on):
        self._ck(lib().wva_pairs_set_pstore(self._h, int(on)))

    def solve_set_ranked(self, on):
        self._ck(lib().wva_solve_set_ranked(self._h, int(on)))

    def type_totals_merge(self, gathered_ptr, n_ranks):
        self._ck(lib().wva_type_totals_merge(self._h, C.c_void_p(int(gathered_ptr)), int(n_ranks)))

    def solve_stats(self):
        v = (C.c_uint64 * 4)()
        self._ck(lib().wva_solve_stats(self._h, v))
        return [int(x) for x in v]

    def solve_greedy_path(self):
        return int(lib().wva_solve_greedy_path(self._h))

    def pairs_set_warp_max(self, n):
        self._ck(lib().wva_pairs_set_warp_max(self._h, int(n)))

    def pair_steps(self):
        v = C.c_uint64(0)
        self._ck(lib().wva_pair_steps(self._h, C.byref(v)))
        return v.value

    def pairs_device(self):
        """Device pointers of the candidate records: dict field -> (address, numpy dtype), plus 'feasible'."""
        dev = abi.AllocSoa()
        fe = C.c_void_p()
        self._ck(lib().wva_pairs_device(self._h, C.byref(dev), C.byref(fe)))
        out = {}
        for name, dt in abi.ALLOC_FIELDS:
            out[name] = (C.cast(getattr(dev, name), C.c_void_p).value, np.dtype(dt))
        out["feasible"] = (fe.value, np.dtype(np.uint8))
        return out

    def pairs_commit(self):
        self._ck(lib().wva_pairs_commit(self._h))

    def analyze_grid(self, r_max, b_max, want_cube=False):
        """Candidate sweep over the shard.  Returns (best[count], cube|None, status|None)."""
        ns = self.count
        best = np.zeros(ns, dtype=abi.GRID_BEST_DTYPE)
        ncand = ns * self.image.A * r_max * b_max
        cube = np.zeros(ncand, dtype=abi.METRICS_DTYPE) if want_cube else None
        status = np.zeros(ncand, dtype=np.uint8) if want_cube else None
        self._ck(lib().wva_analyze_grid(self._h, int(r_max), int(b_max), best.ctypes.data,
                                        cube.ctypes.data if want_cube else None,
                                        status.ctypes.data if want_cube else None))
        return best, cube, status

    def analyze_grid_device(self, r_max, b_max, want_cube=False):
        self._ck(lib().wva_analyze_grid_device(self._h, int(r_max), int(b_max), 1 if want_cube else 0))

    def grid_fetch(self):
        best = np.zeros(self.count, dtype=abi.GRID_BEST_DTYPE)
        self._ck(lib().wva_grid_fetch(self._h, best.ctypes.data))
        return best

    def grid_set_tail_cap(self, cap):
        self._ck(lib().wva_grid_set_tail_cap(self._h, int(cap)))

    def grid_set_pair_winners(self, on):
        """Every later sweep also keeps its best candidate of each (server, accelerator) pair on the device."""
        self._ck(lib().wva_grid_set_pair_winners(self._h, 1 if on else 0))

    def grid_pairs_fetch(self):
        """The sweep's per-pair winners: (AllocArrays[S*A], feasible[S*A]); rows outside the shard are zero."""
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_grid_pairs_fetch(self._h, C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def grid_pairs_size(self, status=None):
        """QueueAnalyzer.Size for every sweep record of the shard at its own batch size: a sized record's
        max_arrv_rate_per_replica becomes the SLO-bound rate.  Returns status[S*A] (0 no record, 1 sized,
        2 Size failed, record unchanged); rows outside the shard keep what `status` held (zeros when None)."""
        status = _status_buffer(status, self.image.S * self.image.A)
        self._ck(lib().wva_grid_pairs_size(self._h, abi.ptr(status, C.c_uint8)))
        return status

    def analyze_scenarios(self, arrival_rpm):
        """What-if Server.Calculate -> unlimited Solve -> AllocateByType for each row of arrival_rpm [L, S] (float32,
        finite; row l replaces every server's arrival rate).  Returns (chosen_acc[L, S], AllocArrays[L*S],
        count[L, T], cost[L, T]); rows of servers outside the shard stay -1 / zero.  The image, pair records,
        solution and totals of the context are left untouched."""
        rates = _scenario_rates(arrival_rpm, self.image.S)
        rc, out = _analyze_scenarios(lib().wva_analyze_scenarios, self._h, self.image.T, rates)
        self._ck(rc)
        return out

    def scenario_pairs_fetch(self, scen):
        """Scenario scen's pair records: (AllocArrays[S*A], feasible[S*A]); rows outside the shard are zero."""
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_scenario_pairs_fetch(self._h, int(scen), C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def grid_list_sizes(self):
        a, b = C.c_int32(0), C.c_int32(0)
        self._ck(lib().wva_grid_list_sizes(self._h, C.byref(a), C.byref(b)))
        return dict(deferred=a.value, literal=b.value)

    def grid_set_fused(self, on):
        self._ck(lib().wva_grid_set_fused(self._h, 1 if on else 0))

    def grid_last_fused(self):
        return int(lib().wva_grid_last_fused(self._h))

    def grid_deferred(self, cap=1 << 22):
        """cube indices (relative to the shard) of the candidates the last sweep slice ran as exact chains."""
        n = C.c_int32(0)
        ids = np.zeros(cap, dtype=np.uint64)
        self._ck(lib().wva_grid_deferred_fetch(self._h, ids.ctypes.data_as(C.POINTER(C.c_uint64)), cap, C.byref(n)))
        return ids[:min(n.value, cap)].copy(), n.value

    def grid_counters(self):
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self._ck(lib().wva_grid_counters(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return dict(steps_executed=a.value, steps_algorithmic=b.value, candidates_ok=c.value)

    # ---- optimize ----------------------------------------------------------------------
    def solve(self, unlimited=True, delayed_best_effort=False, policy=abi.POLICY_NONE, download=True):
        """Solver.Solve.  Returns (chosen_acc[S], AllocArrays[S])."""
        spec = abi.OptimizerSpec(1 if unlimited else 0, 1 if delayed_best_effort else 0, int(policy))
        if not download:
            self._ck(lib().wva_solve(self._h, C.byref(spec), None, None))
            return None
        chosen_acc = np.full(self.image.S, -1, dtype=np.int32)
        chosen = abi.AllocArrays(self.image.S)
        self._ck(lib().wva_solve(self._h, C.byref(spec), abi.ptr(chosen_acc, C.c_int32), C.byref(chosen.c)))
        return chosen_acc, chosen

    def solve_grid(self, unlimited=True, delayed_best_effort=False, policy=abi.POLICY_NONE, download=True):
        """Solver.Solve over the sweep's per-pair winners.  Returns (chosen_acc[S], AllocArrays[S])."""
        spec = abi.OptimizerSpec(1 if unlimited else 0, 1 if delayed_best_effort else 0, int(policy))
        if not download:
            self._ck(lib().wva_solve_grid(self._h, C.byref(spec), None, None))
            return None
        chosen_acc = np.full(self.image.S, -1, dtype=np.int32)
        chosen = abi.AllocArrays(self.image.S)
        self._ck(lib().wva_solve_grid(self._h, C.byref(spec), abi.ptr(chosen_acc, C.c_int32), C.byref(chosen.c)))
        return chosen_acc, chosen

    def allocate_by_type(self, download=True):
        if not download:           # totals stay on the device (type_totals_device)
            self._ck(lib().wva_allocate_by_type(self._h, None, None))
            return None
        count = np.zeros(self.image.T, dtype=np.int64)
        cost = np.zeros(self.image.T, dtype=np.float32)
        self._ck(lib().wva_allocate_by_type(self._h, abi.ptr(count, C.c_int64), abi.ptr(cost, C.c_float)))
        return count, cost

    def type_totals_device(self):
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(lib().wva_type_totals_device(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def solution_time_usec(self):
        return int(lib().wva_solution_time_usec(self._h))

    # ---- pkg/analyzer batched API ----------------------------------------------------
    def queue_analyze(self, cfgs, rates):
        cfgs = np.ascontiguousarray(cfgs, dtype=abi.QUEUE_CONFIG_DTYPE)
        rates = np.ascontiguousarray(rates, dtype=np.float32)
        n = len(cfgs)
        metrics = np.zeros(n, dtype=abi.METRICS_DTYPE)
        status = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_queue_analyze(self._h, n, cfgs.ctypes.data, abi.ptr(rates, C.c_float), metrics.ctypes.data,
                                         abi.ptr(status, C.c_uint8)))
        return metrics, status

    def queue_size(self, cfgs, targets):
        cfgs = np.ascontiguousarray(cfgs, dtype=abi.QUEUE_CONFIG_DTYPE)
        targets = np.ascontiguousarray(targets, dtype=np.float32).reshape(-1)
        n = len(cfgs)
        rates = np.zeros(3 * n, dtype=np.float32)
        achieved = np.zeros(3 * n, dtype=np.float32)
        metrics = np.zeros(n, dtype=abi.METRICS_DTYPE)
        status = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_queue_size(self._h, n, cfgs.ctypes.data, abi.ptr(targets, C.c_float), abi.ptr(rates, C.c_float),
                                      metrics.ctypes.data, abi.ptr(achieved, C.c_float), abi.ptr(status, C.c_uint8)))
        return rates.reshape(n, 3), metrics, achieved.reshape(n, 3), status

    def model_solve(self, K, serv_rate, lambdas, mus):
        """MM1ModelStateDependent(K, serv_rate): consecutive Solve(lambda, mu) calls on one model -> (out[n, 9], p[K+1])"""
        sr = np.ascontiguousarray(serv_rate, dtype=np.float32)
        lam = np.ascontiguousarray(lambdas, dtype=np.float32); mu = np.ascontiguousarray(mus, dtype=np.float32)
        out = np.zeros((len(lam), 9), dtype=np.float32)
        p = np.zeros(int(K) + 1, dtype=np.float64)
        self._ck(lib().wva_model_solve(self._h, int(K), abi.ptr(sr, C.c_float), len(sr), len(lam), abi.ptr(lam, C.c_float),
                                       abi.ptr(mu, C.c_float), abi.ptr(out.reshape(-1), C.c_float), p.ctypes.data_as(C.POINTER(C.c_double))))
        return out, p

    # ---- instrumentation ---------------------------------------------------------------
    def launch_count(self):
        return int(lib().wva_launch_count(self._h))

    def phase_usec(self, phase):
        return int(lib().wva_phase_time_usec(self._h, int(phase)))

    def stream(self):
        """cudaStream_t (as int) all work of this ctx is enqueued on."""
        return int(lib().wva_stream(self._h) or 0)

    def selftest_division(self, seed, n, mode):
        bad = C.c_uint64(0)
        self._ck(lib().wva_selftest_division(self._h, int(seed), int(n), int(mode), C.byref(bad)))
        return bad.value


class Group:
    """wva_group: ONE process driving several GPUs (the shape of the reference's single reconcile goroutine).
    Servers shard over the devices; host outputs have the full extent; totals are global."""

    def __init__(self, devices):
        devs = np.ascontiguousarray(devices, dtype=np.int32)
        self._h = C.c_void_p()
        rc = lib().wva_group_create(abi.ptr(devs, C.c_int32), len(devs), C.byref(self._h))
        if rc != abi.OK:
            raise WvaError(rc, lib().wva_last_error(None).decode())
        self.n = len(devs)
        self.ctxs = [Context(int(devs[i]), _borrowed=lib().wva_group_ctx(self._h, i)) for i in range(self.n)]
        self.image = None

    def close(self):
        if self._h:
            lib().wva_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != abi.OK:
            raise WvaError(rc, lib().wva_group_last_error(self._h).decode())

    def upload(self, image: SystemImage):
        s = image.c_struct()
        self._ck(lib().wva_group_upload(self._h, C.byref(s)))
        self.image = image
        for i, c in enumerate(self.ctxs):
            c.image = image
            c.first = image.S * i // self.n
            c.count = image.S * (i + 1) // self.n - c.first

    def analyze(self, r_max=0, b_max=0, want_cube=False):
        self._ck(lib().wva_group_analyze(self._h, int(r_max), int(b_max), 1 if want_cube else 0))

    def pairs_fetch(self):
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_group_pairs_fetch(self._h, C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def grid_fetch(self):
        best = np.zeros(self.image.S, dtype=abi.GRID_BEST_DTYPE)
        self._ck(lib().wva_group_grid_fetch(self._h, best.ctypes.data))
        return best

    def solve(self, unlimited=True, delayed_best_effort=False, policy=abi.POLICY_NONE, download=True):
        spec = abi.OptimizerSpec(1 if unlimited else 0, 1 if delayed_best_effort else 0, int(policy))
        if not download:
            self._ck(lib().wva_group_solve(self._h, C.byref(spec), None, None))
            return None
        chosen_acc = np.full(self.image.S, -1, dtype=np.int32)
        chosen = abi.AllocArrays(self.image.S)
        self._ck(lib().wva_group_solve(self._h, C.byref(spec), abi.ptr(chosen_acc, C.c_int32), C.byref(chosen.c)))
        return chosen_acc, chosen

    def grid_set_pair_winners(self, on):
        for c in self.ctxs:
            c.grid_set_pair_winners(on)

    def grid_pairs_fetch(self):
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_group_grid_pairs_fetch(self._h, C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def grid_pairs_size(self, status=None):
        """Context.grid_pairs_size on every device (each sizes its shard); status has the full extent S*A"""
        status = _status_buffer(status, self.image.S * self.image.A)
        self._ck(lib().wva_group_grid_pairs_size(self._h, abi.ptr(status, C.c_uint8)))
        return status

    def analyze_scenarios(self, arrival_rpm):
        """Context.analyze_scenarios on every device (each its shard); outputs have the full extent, totals are global"""
        rates = _scenario_rates(arrival_rpm, self.image.S)
        rc, out = _analyze_scenarios(lib().wva_group_analyze_scenarios, self._h, self.image.T, rates)
        self._ck(rc)
        return out

    def scenario_pairs_fetch(self, scen):
        n = self.image.S * self.image.A
        out = abi.AllocArrays(n)
        feasible = np.zeros(n, dtype=np.uint8)
        self._ck(lib().wva_group_scenario_pairs_fetch(self._h, int(scen), C.byref(out.c), abi.ptr(feasible, C.c_uint8)))
        return out, feasible

    def solve_grid(self, unlimited=True, delayed_best_effort=False, policy=abi.POLICY_NONE, download=True):
        spec = abi.OptimizerSpec(1 if unlimited else 0, 1 if delayed_best_effort else 0, int(policy))
        if not download:
            self._ck(lib().wva_group_solve_grid(self._h, C.byref(spec), None, None))
            return None
        chosen_acc = np.full(self.image.S, -1, dtype=np.int32)
        chosen = abi.AllocArrays(self.image.S)
        self._ck(lib().wva_group_solve_grid(self._h, C.byref(spec), abi.ptr(chosen_acc, C.c_int32), C.byref(chosen.c)))
        return chosen_acc, chosen

    def allocate_by_type(self, download=True):
        if not download:
            self._ck(lib().wva_group_allocate_by_type(self._h, None, None))
            return None
        count = np.zeros(self.image.T, dtype=np.int64)
        cost = np.zeros(self.image.T, dtype=np.float32)
        self._ck(lib().wva_group_allocate_by_type(self._h, abi.ptr(count, C.c_int64), abi.ptr(cost, C.c_float)))
        return count, cost
