"""ctypes mirror of include/wva_b200.h (POD structs and constants).

Kept in one place so the product binding (binding.py) and the test-only oracle binding
(oracle/__init__.py) describe the same memory layout.
"""
import ctypes as C

import numpy as np

ABI_VERSION = 1

OK, EINVAL, ECUDA, ESTATE, ENOSOLUTION, ENONFINITE, ECAPACITY = 0, -1, -2, -3, -4, -5, -6

POLICY_NONE, POLICY_PRIORITY_EXHAUSTIVE, POLICY_PRIORITY_ROUND_ROBIN, POLICY_ROUND_ROBIN = 0, 1, 2, 3
POLICY_BY_NAME = {  # SaturatedAllocationPolicyEnum, reference pkg/config/config.go:28-41
    "None": POLICY_NONE,
    "PriorityExhaustive": POLICY_PRIORITY_EXHAUSTIVE,
    "PriorityRoundRobin": POLICY_PRIORITY_ROUND_ROBIN,
    "RoundRobin": POLICY_ROUND_ROBIN,
}

ACC_NONE, ACC_UNKNOWN = -1, -2
COMM_ID_BYTES = 128

CAND_OK, CAND_FEASIBLE = 0, 1
CAND_ERR_PAIR, CAND_ERR_CONFIG, CAND_ERR_RATE_LE0, CAND_ERR_RATE_MAX, CAND_ERR_MODEL = 2, 4, 6, 8, 10

PHASE_UPLOAD, PHASE_PAIRS, PHASE_GRID, PHASE_SOLVE, PHASE_TOTALS, PHASE_GRID_KERNEL, PHASE_GRID_HEAVY, PHASE_GRID_SIZE = 0, 1, 2, 3, 4, 5, 6, 7
PHASE_SCENARIOS = 8
MAX_SCENARIOS = 1024

MAX_QUEUE_TO_BATCH_RATIO = 10
DEFAULT_PRIORITY = 100

f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
u8p = C.POINTER(C.c_uint8)


class SystemSoa(C.Structure):
    _fields_ = [
        ("n_servers", C.c_int32), ("n_accels", C.c_int32), ("n_models", C.c_int32), ("n_types", C.c_int32),
        ("acc_cost", f32p), ("acc_multiplicity", i32p), ("acc_type", i32p),
        ("type_capacity", i64p),
        ("perf_alpha", f32p), ("perf_beta", f32p), ("perf_gamma", f32p), ("perf_delta", f32p),
        ("perf_max_batch", i32p), ("perf_at_tokens", i32p), ("perf_acc_count", i32p), ("perf_valid", u8p),
        ("srv_model", i32p), ("srv_arrival_rpm", f32p), ("srv_in_tokens", i32p), ("srv_out_tokens", i32p),
        ("srv_slo_ttft", f32p), ("srv_slo_itl", f32p), ("srv_slo_tps", f32p), ("srv_target_valid", u8p),
        ("srv_priority", i32p), ("srv_min_replicas", i32p), ("srv_max_batch", i32p), ("srv_keep_acc", u8p),
        ("srv_cur_acc", i32p), ("srv_cur_replicas", i32p), ("srv_cur_cost", f32p),
    ]


# name -> numpy dtype, in struct order, grouped by the dimension each array has
ACC_FIELDS = [("acc_cost", np.float32), ("acc_multiplicity", np.int32), ("acc_type", np.int32)]
TYPE_FIELDS = [("type_capacity", np.int64)]
PERF_FIELDS = [("perf_alpha", np.float32), ("perf_beta", np.float32), ("perf_gamma", np.float32),
               ("perf_delta", np.float32), ("perf_max_batch", np.int32), ("perf_at_tokens", np.int32),
               ("perf_acc_count", np.int32), ("perf_valid", np.uint8)]
SRV_FIELDS = [("srv_model", np.int32), ("srv_arrival_rpm", np.float32), ("srv_in_tokens", np.int32),
              ("srv_out_tokens", np.int32), ("srv_slo_ttft", np.float32), ("srv_slo_itl", np.float32),
              ("srv_slo_tps", np.float32), ("srv_target_valid", np.uint8), ("srv_priority", np.int32),
              ("srv_min_replicas", np.int32), ("srv_max_batch", np.int32), ("srv_keep_acc", np.uint8),
              ("srv_cur_acc", np.int32), ("srv_cur_replicas", np.int32), ("srv_cur_cost", np.float32)]


class AllocSoa(C.Structure):
    _fields_ = [("acc", i32p), ("num_replicas", i64p), ("batch_size", i64p), ("cost", f32p), ("value", f32p),
                ("itl", f32p), ("ttft", f32p), ("rho", f32p), ("max_arrv_rate_per_replica", f32p)]


ALLOC_FIELDS = [("acc", np.int32), ("num_replicas", np.int64), ("batch_size", np.int64), ("cost", np.float32),
                ("value", np.float32), ("itl", np.float32), ("ttft", np.float32), ("rho", np.float32),
                ("max_arrv_rate_per_replica", np.float32)]


class Metrics(C.Structure):
    _fields_ = [("throughput", C.c_float), ("avg_resp_time", C.c_float), ("avg_wait_time", C.c_float),
                ("avg_num_in_serv", C.c_float), ("avg_prefill_time", C.c_float), ("avg_token_time", C.c_float),
                ("max_rate", C.c_float), ("rho", C.c_float)]


METRICS_DTYPE = np.dtype([("throughput", "<f4"), ("avg_resp_time", "<f4"), ("avg_wait_time", "<f4"),
                          ("avg_num_in_serv", "<f4"), ("avg_prefill_time", "<f4"), ("avg_token_time", "<f4"),
                          ("max_rate", "<f4"), ("rho", "<f4")])


class GridBest(C.Structure):
    _fields_ = [("acc", C.c_int32), ("replicas", C.c_int32), ("batch", C.c_int32), ("cost", C.c_float),
                ("value", C.c_float), ("itl", C.c_float), ("ttft", C.c_float), ("rho", C.c_float)]


GRID_BEST_DTYPE = np.dtype([("acc", "<i4"), ("replicas", "<i4"), ("batch", "<i4"), ("cost", "<f4"),
                            ("value", "<f4"), ("itl", "<f4"), ("ttft", "<f4"), ("rho", "<f4")])


class OptimizerSpec(C.Structure):
    _fields_ = [("unlimited", C.c_int32), ("delayed_best_effort", C.c_int32), ("saturation_policy", C.c_int32)]


class QueueConfig(C.Structure):
    _fields_ = [("max_batch_size", C.c_int32), ("max_queue_size", C.c_int32), ("alpha", C.c_float),
                ("beta", C.c_float), ("gamma", C.c_float), ("delta", C.c_float),
                ("avg_input_tokens", C.c_int32), ("avg_output_tokens", C.c_int32)]


QUEUE_CONFIG_DTYPE = np.dtype([("max_batch_size", "<i4"), ("max_queue_size", "<i4"), ("alpha", "<f4"),
                               ("beta", "<f4"), ("gamma", "<f4"), ("delta", "<f4"),
                               ("avg_input_tokens", "<i4"), ("avg_output_tokens", "<i4")])

assert C.sizeof(Metrics) == METRICS_DTYPE.itemsize == 32
assert C.sizeof(GridBest) == GRID_BEST_DTYPE.itemsize == 32
assert C.sizeof(QueueConfig) == QUEUE_CONFIG_DTYPE.itemsize == 32


def ptr(arr, ctype):
    """Typed pointer to a C-contiguous numpy array (caller keeps the array alive)."""
    assert arr.flags["C_CONTIGUOUS"]
    return arr.ctypes.data_as(C.POINTER(ctype))


_CT = {np.dtype(np.float32): C.c_float, np.dtype(np.int32): C.c_int32, np.dtype(np.int64): C.c_int64,
       np.dtype(np.uint8): C.c_uint8}


class AllocArrays:
    """Caller-owned wva_alloc_soa of length n backed by numpy arrays."""

    def __init__(self, n):
        self.n = int(n)
        for name, dt in ALLOC_FIELDS:
            setattr(self, name, np.zeros(self.n, dtype=dt))
        self.c = AllocSoa(*[ptr(getattr(self, name), _CT[np.dtype(dt)]) for name, dt in ALLOC_FIELDS])

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in ALLOC_FIELDS}

    def equal_bits(self, other, mask=None):
        """Bit-exact comparison (floats compared through their integer views)."""
        for name, dt in ALLOC_FIELDS:
            a, b = getattr(self, name), getattr(other, name)
            if mask is not None:
                a, b = a[mask], b[mask]
            if np.dtype(dt) == np.float32:
                # NaN payloads are not part of the contract: an invalid operation (Inf - Inf) yields 0xFFC00000 on amd64
                # (the reference's platform) and 0x7FFFFFFF on NVIDIA GPUs; every other value is compared bit for bit
                both_nan = np.isnan(a) & np.isnan(b)
                a, b = np.where(both_nan, np.uint32(0), a.view(np.uint32)), np.where(both_nan, np.uint32(0), b.view(np.uint32))
            if not np.array_equal(a, b):
                return False, name
        return True, None
