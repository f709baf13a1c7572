"""ctypes binding of include/povar_b200.h (libpovar_b200.so).

This is plumbing for the tests, the benchmark and Python callers; the product is the shared
library.  There is no Python or CPU implementation behind these calls: if the library is
missing, import fails; if there is no CUDA device, `povar_create` returns POVAR_ERR_NO_DEVICE.
The logic of its own is argument checking and the conversions around the calls: HostProblem's
canonical order and shards, DeviceProblem's checks of torch tensors and its shards (torch is
imported only where a DeviceProblem or a device-state call needs it).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# POVAR_LIB: a tuning build of the same library (povar_b200.build.build(defines=..., suffix=...))
LIB_PATH = os.environ.get("POVAR_LIB") or os.path.join(_HERE, "lib", "libpovar_b200.so")

# status codes / enums (include/povar_b200.h)
OK = 0
NUM_NONFINITE_INC = 1
NUM_LINEARIZATION = 2
ERR_INVALID, ERR_CUDA, ERR_NCCL, ERR_NO_DEVICE, ERR_IO, ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
PCG, POWER_SCHUR_COMPLEMENT, POWER_VARPROJ, CHOLESKY = 0, 1, 2, 3
RIPOBA, RIPCG = 0, 1
NORM_NONE, NORM_HUBER, NORM_CAUCHY = 0, 1, 2
STATE_POSE, STATE_JOINT = 0, 1

STEP1_NAMES = {"PCG": PCG, "POWER_SCHUR_COMPLEMENT": POWER_SCHUR_COMPLEMENT,
               "POWER_BUNDLE_ADJUSTMENT": POWER_SCHUR_COMPLEMENT, "POWER_VARPROJ": POWER_VARPROJ,
               "CHOLESKY": CHOLESKY}
STEP2_NAMES = {"RIPOBA": RIPOBA, "RIPCG": RIPCG}
NORM_NAMES = {"NONE": NORM_NONE, "HUBER": NORM_HUBER, "CAUCHY": NORM_CAUCHY}


class Options(C.Structure):
    _fields_ = [
        ("solver_type_step_1", C.c_int32), ("solver_type_step_2", C.c_int32),
        ("robust_norm", C.c_int32), ("optimized_cost", C.c_int32),
        ("huber_parameter", C.c_double), ("alpha", C.c_double),
        ("max_num_iterations_step_1", C.c_int32), ("max_num_iterations_step_2", C.c_int32),
        ("min_relative_decrease", C.c_double), ("initial_trust_region_radius", C.c_double),
        ("min_trust_region_radius", C.c_double), ("max_trust_region_radius", C.c_double),
        ("min_linear_solver_iterations", C.c_int32), ("max_linear_solver_iterations", C.c_int32),
        ("eta", C.c_double), ("r_tolerance", C.c_double), ("jacobi_scaling_epsilon", C.c_double),
        ("function_tolerance", C.c_double), ("power_sc_iterations", C.c_int32),
        ("verbosity_level", C.c_int32), ("initial_vee", C.c_double), ("vee_factor", C.c_double),
    ]


class ProblemDesc(C.Structure):
    _fields_ = [
        ("num_cams", C.c_int32), ("num_lms", C.c_int32), ("num_obs", C.c_int64),
        ("lm_ptr", C.POINTER(C.c_int64)), ("obs_cam", C.POINTER(C.c_int32)),
        ("obs_uv", C.POINTER(C.c_double)), ("cam_P", C.POINTER(C.c_double)),
    ]


class DeviceProblemDesc(C.Structure):
    _fields_ = [
        ("num_cams", C.c_int32), ("num_lms", C.c_int32), ("num_obs", C.c_int64),
        ("lm_begin", C.c_int32), ("lm_end", C.c_int32),
        ("obs_cam", C.c_void_p), ("obs_lm", C.c_void_p), ("obs_uv", C.c_void_p), ("cam_P", C.c_void_p),
        ("stream", C.c_void_p),
    ]


class ResidualInfo(C.Structure):
    _fields_ = [
        ("num_obs_all", C.c_int64), ("error_all", C.c_double), ("residual_sum_all", C.c_double),
        ("num_obs_valid", C.c_int64), ("error_valid", C.c_double), ("residual_sum_valid", C.c_double),
        ("is_numerically_valid", C.c_int32),
    ]


class CommDesc(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world_size", C.c_int32), ("device", C.c_int32),
                ("nccl_id", C.c_uint8 * 128)]


class BalData(C.Structure):
    _fields_ = [
        ("num_cams", C.c_int32), ("num_lms", C.c_int32), ("num_obs", C.c_int64),
        ("lm_ptr", C.POINTER(C.c_int64)), ("obs_cam", C.POINTER(C.c_int32)),
        ("obs_uv", C.POINTER(C.c_double)), ("cam_params", C.POINTER(C.c_double)),
    ]


class Iteration(C.Structure):
    _fields_ = [
        ("step", C.c_int32), ("iteration", C.c_int32), ("step_is_valid", C.c_int32),
        ("step_is_successful", C.c_int32), ("cost", C.c_double), ("cost_valid", C.c_double),
        ("trial_cost", C.c_double), ("num_obs_valid", C.c_int64), ("relative_decrease", C.c_double),
        ("trust_region_radius", C.c_double), ("linear_solver_iterations", C.c_int32),
        ("iteration_time", C.c_double), ("cumulative_time", C.c_double),
        ("residual_evaluation_time", C.c_double), ("jacobian_evaluation_time", C.c_double),
        ("prepare_time", C.c_double), ("solve_reduced_system_time", C.c_double),
        ("back_substitution_time", C.c_double),
        ("residual_mean", C.c_double), ("residual_valid_mean", C.c_double),
    ]


class BaLogInfo(C.Structure):
    _fields_ = [("input_path", C.c_char_p), ("num_cams", C.c_int32), ("num_lms", C.c_int32), ("num_obs", C.c_int64),
                ("lm_ptr", C.POINTER(C.c_int64)), ("load_time", C.c_double), ("num_gpus", C.c_int32)]


class SolveSummary(C.Structure):
    _fields_ = [
        ("num_iterations", C.c_int32), ("termination_type_step_1", C.c_int32),
        ("termination_type_step_2", C.c_int32), ("num_successful_steps", C.c_int32),
        ("num_unsuccessful_steps", C.c_int32), ("initial_cost", C.c_double), ("final_cost", C.c_double),
        ("total_time", C.c_double), ("step1_time", C.c_double), ("step2_time", C.c_double),
        ("power_terms", C.c_int64), ("power_series_time", C.c_double), ("message", C.c_char * 256),
    ]


class PhaseTimes(C.Structure):
    _fields_ = [("residual_evaluation_time", C.c_double), ("jacobian_evaluation_time", C.c_double),
                ("prepare_time", C.c_double), ("solve_reduced_system_time", C.c_double),
                ("back_substitution_time", C.c_double)]


# every symbol include/povar_b200.h declares: (restype, argtypes)
_H = C.c_void_p
_DP = C.POINTER(C.c_double)
SIGNATURES = {
    "povar_abi_version": (C.c_int, []),
    "povar_abi_sizeof": (C.c_int64, [C.c_int32]),
    "povar_options_default": (None, [C.POINTER(Options)]),
    "povar_bal_read": (C.c_int, [C.c_char_p, C.POINTER(BalData), C.c_char_p, C.c_size_t]),
    "povar_bal_free": (None, [C.POINTER(BalData)]),
    "povar_canonical_order": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_int32),
                                        C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "povar_partition_landmarks": (C.c_int, [C.c_int32, C.POINTER(C.c_int64), C.c_int32, C.POINTER(C.c_int32)]),
    "povar_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "povar_comm_host_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "povar_get_timings": (C.c_int, [_H, C.POINTER(PhaseTimes)]),
    "povar_reset_timings": (C.c_int, [_H]),
    "povar_create": (C.c_int, [C.POINTER(ProblemDesc), C.POINTER(Options), C.POINTER(CommDesc), C.POINTER(_H)]),
    "povar_create_device": (C.c_int, [C.POINTER(DeviceProblemDesc), C.POINTER(Options), C.POINTER(CommDesc),
                                      C.POINTER(_H)]),
    "povar_destroy": (None, [_H]),
    "povar_last_error": (C.c_char_p, [_H]),
    "povar_init_varproj": (C.c_int, [_H, C.c_double]),
    "povar_cost_pose": (C.c_int, [_H, C.c_double, C.POINTER(ResidualInfo)]),
    "povar_cost_homogeneous": (C.c_int, [_H, C.POINTER(ResidualInfo)]),
    "povar_linearize_pose": (C.c_int, [_H, C.c_double]),
    "povar_linearize_homogeneous": (C.c_int, [_H]),
    "povar_solve_pose": (C.c_int, [_H, C.c_double, _DP, C.POINTER(C.c_int32)]),
    "povar_solve_joint": (C.c_int, [_H, C.c_double, _DP, C.POINTER(C.c_int32)]),
    "povar_apply_pose": (C.c_int, [_H, C.c_double, _DP]),
    "povar_apply_joint": (C.c_int, [_H, _DP]),
    "povar_backup": (C.c_int, [_H, C.c_int32]),
    "povar_restore": (C.c_int, [_H, C.c_int32]),
    "povar_to_homogeneous": (C.c_int, [_H]),
    "povar_normalize_joint": (C.c_int, [_H]),
    "povar_get_state": (C.c_int, [_H, C.c_int32, _DP, _DP]),
    "povar_set_state": (C.c_int, [_H, C.c_int32, _DP, _DP]),
    "povar_get_state_device": (C.c_int, [_H, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "povar_set_state_device": (C.c_int, [_H, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "povar_bundle_adjust": (C.c_int, [_H, C.POINTER(Options), C.POINTER(Iteration), C.c_int32,
                                      C.POINTER(SolveSummary)]),
    "povar_bundle_adjust_async": (C.c_int, [_H, C.POINTER(Options), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "povar_comm_finalize": (C.c_int, []),
    "povar_debug_read": (C.c_int64, [_H, C.c_char_p, _DP, C.c_int64]),
    "povar_right_mul_e0": (C.c_int, [_H, C.c_int32, _DP, _DP]),
    "povar_bench_power_terms": (C.c_int, [_H, C.c_int32, C.c_int32, _DP]),
    "povar_bench_power_kernels": (C.c_int, [_H, C.c_int32, C.c_int32, _DP]),
    "povar_launch_count": (C.c_int64, [_H]),
    "povar_bal_create_dataset": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int64, C.c_char_p, C.c_size_t]),
    "povar_peer_exchange_active": (C.c_int, [_H]),
    "povar_debug_set_window": (C.c_int, [_H, C.c_int32]),
    "povar_debug_cholesky": (C.c_int, [C.c_int32, _DP, _DP, _DP, C.POINTER(C.c_int32)]),
    "povar_debug_set_cholesky_storage": (C.c_int, [_H, C.c_int32]),
    "povar_debug_sparse_cholesky": (C.c_int, [C.c_int32, C.c_int32, _DP, _DP, _DP, C.POINTER(C.c_int32),
                                              C.POINTER(C.c_int64)]),
    "povar_debug_cholesky_symbolic": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                                C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "povar_write_ba_log": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "povar_debug_sell_layout": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_int32,
                                          C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                          C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "povar_debug_sell_max_degree": (C.c_int, [C.c_int64, C.c_int32]),
    "povar_debug_landmark_plan": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.c_int32,
                                            C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32),
                                            C.POINTER(C.c_int32)]),
    "povar_debug_walk_trace": (C.c_int, [C.POINTER(C.c_uint64), C.c_int32]),
    "povar_cuda_stream": (C.c_void_p, [_H]),
}

_lib = None


def load():
    """dlopen libpovar_b200.so (fails loudly if it was not built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m povar_b200.build` "
                              "(the CUDA library is the product; there is no fallback)")
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def default_options(**overrides) -> Options:
    lib = load()
    o = Options()
    lib.povar_options_default(C.byref(o))
    for k, v in overrides.items():
        if not hasattr(o, k):
            raise AttributeError(f"unknown option {k}")
        setattr(o, k, v)
    return o


def _dp(a: np.ndarray):
    return a.ctypes.data_as(_DP)


class PovarError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"povar error {code}: {msg}")
        self.code = code


class HostProblem:
    """A BAL problem in canonical order on the host (numpy views of povar_bal_read's output or
    arrays built from a generator)."""

    def __init__(self, num_cams, num_lms, lm_ptr, obs_cam, obs_uv, cam_params):
        self.num_cams = int(num_cams)
        self.num_lms = int(num_lms)
        self.lm_ptr = np.ascontiguousarray(lm_ptr, dtype=np.int64)
        self.obs_cam = np.ascontiguousarray(obs_cam, dtype=np.int32)
        self.obs_uv = np.ascontiguousarray(obs_uv, dtype=np.float64).reshape(-1, 2)
        self.cam_params = np.ascontiguousarray(cam_params, dtype=np.float64).reshape(self.num_cams, -1)
        self.cam_P = np.ascontiguousarray(self.cam_params[:, :12])

    @property
    def num_obs(self):
        return int(self.obs_cam.shape[0])

    @staticmethod
    def read(path: str) -> "HostProblem":
        lib = load()
        data = BalData()
        err = C.create_string_buffer(512)
        rc = lib.povar_bal_read(path.encode(), C.byref(data), err, 512)
        if rc != OK:
            raise PovarError(rc, err.value.decode())
        try:
            L, N, Cn = data.num_lms, data.num_obs, data.num_cams
            hp = HostProblem(
                Cn, L,
                np.ctypeslib.as_array(data.lm_ptr, shape=(L + 1,)).copy(),
                np.ctypeslib.as_array(data.obs_cam, shape=(N,)).copy(),
                np.ctypeslib.as_array(data.obs_uv, shape=(N, 2)).copy(),
                np.ctypeslib.as_array(data.cam_params, shape=(Cn, 15)).copy())
        finally:
            lib.povar_bal_free(C.byref(data))
        return hp

    @staticmethod
    def from_unordered(num_cams, num_lms, obs_cam, obs_lm, obs_xy_file, cam_params) -> "HostProblem":
        """canonical order + y flip through the library (povar_canonical_order)."""
        lib = load()
        cam = np.ascontiguousarray(obs_cam, dtype=np.int32)
        lm = np.ascontiguousarray(obs_lm, dtype=np.int32)
        n = cam.shape[0]
        perm = np.empty(n, dtype=np.int64)
        lm_ptr = np.empty(num_lms + 1, dtype=np.int64)
        rc = lib.povar_canonical_order(num_cams, num_lms, n, cam.ctypes.data_as(C.POINTER(C.c_int32)),
                                       lm.ctypes.data_as(C.POINTER(C.c_int32)),
                                       perm.ctypes.data_as(C.POINTER(C.c_int64)),
                                       lm_ptr.ctypes.data_as(C.POINTER(C.c_int64)))
        if rc != OK:
            raise PovarError(rc, "povar_canonical_order: duplicate or out-of-range observation")
        uv = np.array(obs_xy_file, dtype=np.float64)[perm]
        uv[:, 1] = -uv[:, 1]
        return HostProblem(num_cams, num_lms, lm_ptr, cam[perm], uv, cam_params)

    def shard(self, rank: int, world: int) -> "HostProblem":
        lib = load()
        bounds = np.empty(world + 1, dtype=np.int32)
        lib.povar_partition_landmarks(self.num_lms, self.lm_ptr.ctypes.data_as(C.POINTER(C.c_int64)), world,
                                      bounds.ctypes.data_as(C.POINTER(C.c_int32)))
        lb, le = int(bounds[rank]), int(bounds[rank + 1])
        ob, oe = int(self.lm_ptr[lb]), int(self.lm_ptr[le])
        hp = HostProblem(self.num_cams, le - lb, self.lm_ptr[lb:le + 1] - ob, self.obs_cam[ob:oe],
                         self.obs_uv[ob:oe], self.cam_params)
        hp.lm_begin, hp.lm_end = lb, le
        return hp


class DeviceProblem:
    """A BAL problem whose observations live on the GPU as torch CUDA tensors, in any order: the library orders
    them on the device (povar_create_device).  cam_P [C, 12] or [C, 3, 4] float64; obs_cam, obs_lm [N] int32;
    obs_uv [N, 2] float64 after the y flip; all contiguous, on one CUDA device.  num_lms: landmarks of the whole
    problem (default: max(obs_lm) + 1, which reads one number back); lm_range: the landmarks [begin, end) this
    handle takes (default: all).  num_lms is that of the range, num_obs the length of the list."""

    def __init__(self, cam_P, obs_cam, obs_lm, obs_uv, num_lms=None, lm_range=None):
        import torch
        ts = {"cam_P": cam_P, "obs_cam": obs_cam, "obs_lm": obs_lm, "obs_uv": obs_uv}
        for name, t in ts.items():
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"DeviceProblem: {name} must be a torch tensor")
            if t.dtype != (torch.int32 if name in ("obs_cam", "obs_lm") else torch.float64):
                raise ValueError(f"DeviceProblem: {name} has dtype {t.dtype}")
            if not t.is_contiguous():
                raise ValueError(f"DeviceProblem: {name} must be contiguous")
        n = obs_cam.shape[0] if obs_cam.dim() == 1 else -1
        if obs_cam.dim() != 1 or tuple(obs_lm.shape) != (n,) or tuple(obs_uv.shape) != (n, 2):
            raise ValueError("DeviceProblem: obs_cam, obs_lm must be [N] and obs_uv [N, 2]")
        if cam_P.dim() == 0 or cam_P.shape[0] == 0 or cam_P.numel() != cam_P.shape[0] * 12:
            raise ValueError("DeviceProblem: cam_P must be [C, 12] or [C, 3, 4] with C > 0")
        if num_lms is not None and int(num_lms) < 0:
            raise ValueError(f"DeviceProblem: num_lms = {num_lms}")
        if lm_range is not None:
            lb, le = int(lm_range[0]), int(lm_range[1])
            if not 0 <= lb <= le or (num_lms is not None and le > int(num_lms)):
                raise ValueError(f"DeviceProblem: landmark range [{lb}, {le}) is not inside [0, num_lms = {num_lms}]")
        for name, t in ts.items():
            if t.device.type != "cuda":
                raise ValueError(f"DeviceProblem: {name} must be a CUDA tensor (it is on {t.device})")
            if t.device != cam_P.device:
                raise ValueError(f"DeviceProblem: {name} is on {t.device}, cam_P on {cam_P.device}")
        if num_lms is None:
            num_lms = int(obs_lm.max().item()) + 1 if n > 0 else 0
        num_lms = int(num_lms)
        lb, le = (0, num_lms) if lm_range is None else (int(lm_range[0]), int(lm_range[1]))
        if le > num_lms:
            raise ValueError(f"DeviceProblem: landmark range [{lb}, {le}) is not inside [0, num_lms = {num_lms}]")
        self.cam_P, self.obs_cam, self.obs_lm, self.obs_uv = cam_P, obs_cam, obs_lm, obs_uv
        self.num_cams = int(cam_P.shape[0])
        self.num_lms_total = num_lms
        self.lm_begin, self.lm_end = lb, le
        self.num_lms = le - lb
        self.num_obs = int(n)
        self.device = cam_P.device

    def shard(self, rank: int, world: int) -> "DeviceProblem":
        """The landmark range of `rank` out of `world` (povar_partition_landmarks on the per-landmark counts of the
        whole list); every rank keeps the whole list."""
        import torch
        counts = torch.bincount(self.obs_lm.long(), minlength=self.num_lms_total)[:self.num_lms_total]
        lm_ptr = np.zeros(self.num_lms_total + 1, dtype=np.int64)
        lm_ptr[1:] = torch.cumsum(counts, 0).cpu().numpy()
        bounds = np.empty(world + 1, dtype=np.int32)
        rc = load().povar_partition_landmarks(self.num_lms_total, lm_ptr.ctypes.data_as(C.POINTER(C.c_int64)), world,
                                              bounds.ctypes.data_as(C.POINTER(C.c_int32)))
        if rc != OK:
            raise PovarError(rc, "povar_partition_landmarks failed")
        return DeviceProblem(self.cam_P, self.obs_cam, self.obs_lm, self.obs_uv, self.num_lms_total,
                             (int(bounds[rank]), int(bounds[rank + 1])))


class Solver:
    """Handle wrapper with the reference's Linearizor method names
    (/root/reference/src/rootba_povar/solver/linearizor.hpp:47-82)."""

    def __init__(self, problem: HostProblem | DeviceProblem, options: Options | None = None,
                 comm: CommDesc | None = None):
        self.lib = load()
        self.problem = problem
        self.options = options if options is not None else default_options()
        self.device_index = comm.device if comm else 0   # the handle's CUDA device
        h = _H()
        if isinstance(problem, DeviceProblem):
            import torch
            with torch.cuda.device(problem.device):
                desc = DeviceProblemDesc(problem.num_cams, problem.num_lms_total, problem.num_obs, problem.lm_begin,
                                         problem.lm_end, problem.obs_cam.data_ptr(), problem.obs_lm.data_ptr(),
                                         problem.obs_uv.data_ptr(), problem.cam_P.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream)
            rc = self.lib.povar_create_device(C.byref(desc), C.byref(self.options), C.byref(comm) if comm else None,
                                              C.byref(h))
        else:
            desc = ProblemDesc()
            desc.num_cams = problem.num_cams
            desc.num_lms = problem.num_lms
            desc.num_obs = problem.num_obs
            desc.lm_ptr = problem.lm_ptr.ctypes.data_as(C.POINTER(C.c_int64))
            desc.obs_cam = problem.obs_cam.ctypes.data_as(C.POINTER(C.c_int32))
            desc.obs_uv = problem.obs_uv.ctypes.data_as(_DP)
            desc.cam_P = problem.cam_P.ctypes.data_as(_DP)
            rc = self.lib.povar_create(C.byref(desc), C.byref(self.options), C.byref(comm) if comm else None,
                                       C.byref(h))
        if rc != OK:
            raise PovarError(rc, self.lib.povar_last_error(None).decode())
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.povar_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, allow=()):
        if rc != OK and rc not in allow:
            raise PovarError(rc, self.lib.povar_last_error(self.h).decode())
        return rc

    # --- Linearizor interface
    def initialize_varproj_lm_pOSE(self, alpha):
        self._check(self.lib.povar_init_varproj(self.h, alpha))

    def compute_error_pOSE(self, alpha) -> ResidualInfo:
        ri = ResidualInfo()
        self._check(self.lib.povar_cost_pose(self.h, alpha, C.byref(ri)))
        return ri

    def compute_error_homogeneous(self) -> ResidualInfo:
        ri = ResidualInfo()
        self._check(self.lib.povar_cost_homogeneous(self.h, C.byref(ri)))
        return ri

    def linearize_pOSE(self, alpha):
        return self._check(self.lib.povar_linearize_pose(self.h, alpha), allow=(NUM_LINEARIZATION,))

    def linearize_projective_space_homogeneous(self):
        return self._check(self.lib.povar_linearize_homogeneous(self.h), allow=(NUM_LINEARIZATION,))

    def solve(self, lam):
        """-> (inc [C,12], linear_solver_iterations, status)"""
        inc = np.empty((self.problem.num_cams, 12))
        its = C.c_int32(0)
        rc = self._check(self.lib.povar_solve_pose(self.h, lam, _dp(inc), C.byref(its)),
                         allow=(NUM_NONFINITE_INC,))
        return inc, its.value, rc

    def solve_joint(self, lam):
        inc = np.empty((self.problem.num_cams, 11))
        its = C.c_int32(0)
        rc = self._check(self.lib.povar_solve_joint(self.h, lam, _dp(inc), C.byref(its)),
                         allow=(NUM_NONFINITE_INC,))
        return inc, its.value, rc

    def apply(self, alpha) -> float:
        l = C.c_double(0)
        self._check(self.lib.povar_apply_pose(self.h, alpha, C.byref(l)))
        return l.value

    def apply_joint(self) -> float:
        l = C.c_double(0)
        self._check(self.lib.povar_apply_joint(self.h, C.byref(l)))
        return l.value

    # --- caller-side state handling of the reference
    def backup(self, which):
        self._check(self.lib.povar_backup(self.h, which))

    def restore(self, which):
        self._check(self.lib.povar_restore(self.h, which))

    def to_homogeneous(self):
        self._check(self.lib.povar_to_homogeneous(self.h))

    def normalize_joint(self):
        self._check(self.lib.povar_normalize_joint(self.h))

    def get_state(self, which, out=None):
        """`out`: (P, X) buffers of the caller (C-contiguous float64, e.g. page-locked) to read the state into."""
        w = 4 if which == STATE_JOINT else 3
        if out is not None:
            P, X = out
            if (P.dtype != np.float64 or X.dtype != np.float64 or not P.flags.c_contiguous or not X.flags.c_contiguous
                    or P.size != self.problem.num_cams * 12 or X.size != self.problem.num_lms * w):
                raise ValueError("get_state: out buffers must be C-contiguous float64 of the state's size")
        else:
            P = np.empty((self.problem.num_cams, 3, 4))
            X = np.empty((self.problem.num_lms, w))
        self._check(self.lib.povar_get_state(self.h, which, _dp(P), _dp(X)))
        return P, X

    def set_state(self, which, P=None, X=None):
        Pc = np.ascontiguousarray(P, dtype=np.float64) if P is not None else None
        Xc = np.ascontiguousarray(X, dtype=np.float64) if X is not None else None
        self._check(self.lib.povar_set_state(self.h, which, _dp(Pc) if Pc is not None else None,
                                             _dp(Xc) if Xc is not None else None))

    def get_state_device(self, which):
        """-> (P [C, 3, 4], X [L, 3|4]) float64 tensors on the handle's device, written on the current torch stream
        (no host synchronisation)."""
        import torch
        dev = torch.device("cuda", self.device_index)
        P = torch.empty((self.problem.num_cams, 3, 4), dtype=torch.float64, device=dev)
        X = torch.empty((self.problem.num_lms, 4 if which == STATE_JOINT else 3), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream().cuda_stream
        self._check(self.lib.povar_get_state_device(self.h, which, P.data_ptr(), X.data_ptr(), stream))
        return P, X

    def set_state_device(self, which, P=None, X=None):
        """State from float64 CUDA tensors (P [C, 3, 4] or [C, 12], X [L, 3|4]) on the current torch stream."""
        import torch
        w = 4 if which == STATE_JOINT else 3
        want = {"P": self.problem.num_cams * 12, "X": self.problem.num_lms * w}
        dev = None
        for name, t in (("P", P), ("X", X)):
            if t is None:
                continue
            if (not isinstance(t, torch.Tensor) or t.device.type != "cuda" or t.dtype != torch.float64
                    or not t.is_contiguous() or t.numel() != want[name]):
                raise ValueError(f"set_state_device: {name} must be a contiguous float64 CUDA tensor of "
                                 f"{want[name]} elements")
            dev = t.device
        if dev is None:
            return
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream().cuda_stream
        self._check(self.lib.povar_set_state_device(self.h, which, P.data_ptr() if P is not None else None,
                                                    X.data_ptr() if X is not None else None, stream))

    # --- driver and instrumentation
    def bundle_adjust(self, options: Options | None = None):
        opt = options if options is not None else self.options
        cap = opt.max_num_iterations_step_1 + opt.max_num_iterations_step_2 + 4
        its = (Iteration * cap)()
        summary = SolveSummary()
        rc = self.lib.povar_bundle_adjust(self.h, C.byref(opt), its, cap, C.byref(summary))
        if rc != OK:
            raise PovarError(rc, summary.message.decode() + " / " + self.lib.povar_last_error(self.h).decode())
        return [its[i] for i in range(summary.num_iterations)], summary

    def bundle_adjust_async(self, options: Options | None = None) -> "AsyncSolve":
        """bundle_adjust enqueued on the current torch stream of the handle's device, without a host
        synchronisation; `.result()` of the returned object gives what bundle_adjust returns."""
        import torch
        opt = options if options is not None else self.options
        if not isinstance(opt, Options):
            raise ValueError("bundle_adjust_async: options must be a capi.Options")
        if opt.max_num_iterations_step_1 < 0 or opt.max_num_iterations_step_2 < 0:
            raise ValueError("bundle_adjust_async: negative maximum number of iterations")
        if not getattr(self, "h", None):
            raise ValueError("bundle_adjust_async: the solver is closed")
        cap = opt.max_num_iterations_step_1 + opt.max_num_iterations_step_2 + 2
        dev = torch.device("cuda", self.device_index)
        log = torch.empty(cap * C.sizeof(Iteration), dtype=torch.uint8, device=dev)
        summary = torch.empty(C.sizeof(SolveSummary), dtype=torch.uint8, device=dev)
        status = torch.empty(1, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream()
        self._check(self.lib.povar_bundle_adjust_async(self.h, C.byref(opt), log.data_ptr(), cap, summary.data_ptr(),
                                                       status.data_ptr(), stream.cuda_stream))
        return AsyncSolve(self, log, summary, status, stream)

    def debug_read(self, name: str) -> np.ndarray:
        n = self.lib.povar_debug_read(self.h, name.encode(), None, 0)
        if n < 0:
            raise PovarError(n, self.lib.povar_last_error(self.h).decode())
        out = np.empty(int(n))
        self.lib.povar_debug_read(self.h, name.encode(), _dp(out), n)
        return out

    def debug_count(self, name: str) -> int:
        """Number of elements of a device array (no copy)."""
        n = self.lib.povar_debug_read(self.h, name.encode(), None, 0)
        if n < 0:
            raise PovarError(n, self.lib.povar_last_error(self.h).decode())
        return int(n)

    def right_mul_e0(self, which, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty_like(x)
        self._check(self.lib.povar_right_mul_e0(self.h, which, _dp(x), _dp(out)))
        return out

    def bench_power_terms(self, which, terms: int) -> float:
        s = C.c_double(0)
        self._check(self.lib.povar_bench_power_terms(self.h, which, terms, C.byref(s)))
        return s.value

    def bench_power_kernels(self, which, reps: int) -> np.ndarray:
        out = np.zeros(4)
        self._check(self.lib.povar_bench_power_kernels(self.h, which, reps, _dp(out)))
        return out

    def cuda_stream(self) -> int:
        """cudaStream_t of the handle as an integer (for torch.cuda.ExternalStream)."""
        return int(self.lib.povar_cuda_stream(self.h) or 0)

    def peer_exchange_active(self) -> bool:
        return bool(self.lib.povar_peer_exchange_active(self.h))

    def debug_set_window(self, cams: int) -> None:
        self._check(self.lib.povar_debug_set_window(self.h, cams))

    def debug_set_cholesky_storage(self, mode: int) -> None:
        """CHOLESKY storage of S: 0 dense while it fits under 96 GB, tile-sparse beyond; 1 tile-sparse always."""
        self._check(self.lib.povar_debug_set_cholesky_storage(self.h, mode))

    def launch_count(self) -> int:
        return int(self.lib.povar_launch_count(self.h))

    def timings(self) -> PhaseTimes:
        """CUDA-event phase times accumulated since the last reset_timings (povar_get_timings)"""
        t = PhaseTimes()
        self._check(self.lib.povar_get_timings(self.h, C.byref(t)))
        return t

    def reset_timings(self) -> None:
        self._check(self.lib.povar_reset_timings(self.h))


class AsyncSolve:
    """An enqueued solve (Solver.bundle_adjust_async): the log, the summary and the status in device tensors, written
    on `stream` when the solve ends."""

    def __init__(self, solver, log, summary, status, stream):
        self.solver, self.log, self.summary, self.status, self.stream = solver, log, summary, status, stream

    def result(self):
        """Synchronises the stream and decodes -> (list[Iteration], SolveSummary); PovarError on a failed solve."""
        self.stream.synchronize()
        summary = SolveSummary.from_buffer_copy(self.summary.cpu().numpy().tobytes())
        raw = self.log.cpu().numpy().tobytes()
        n = min(summary.num_iterations, len(raw) // C.sizeof(Iteration))
        its = [Iteration.from_buffer_copy(raw, i * C.sizeof(Iteration)) for i in range(n)]
        rc = int(self.status.cpu()[0])
        if rc != OK:
            raise PovarError(rc, summary.message.decode())
        return its, summary


def write_ba_log(path: str, hp: "HostProblem", options, iterations, summary, input_path: str = "", load_time=0.0,
                 num_gpus: int = 1) -> None:
    """ba_log.json with the reference's key set (what `bal --log-log-path` writes) from a solve's records."""
    lib = load()
    lp = np.ascontiguousarray(hp.lm_ptr, dtype=np.int64)
    info = BaLogInfo(input_path.encode(), hp.num_cams, hp.num_lms, hp.num_obs,
                     lp.ctypes.data_as(C.POINTER(C.c_int64)), load_time, num_gpus)
    arr = (Iteration * max(len(iterations), 1))(*iterations)
    rc = lib.povar_write_ba_log(path.encode(), C.byref(info), C.byref(options), arr, len(iterations), C.byref(summary))
    if rc != OK:
        raise PovarError(rc, "povar_write_ba_log failed")


def sell_max_degree(num_obs: int, sms: int = 148) -> int:
    """Largest degree of a landmark of the sliced-ELL set for a shard of num_obs observations."""
    return int(load().povar_debug_sell_max_degree(num_obs, sms))


def sell_layout(hp: "HostProblem", threads: int = 0, max_deg: int = 0):
    """(slice_ptr, sell_lm, long_lms) of the sliced-ELL landmark order of `hp` (max_deg = 0: landmarks with up to 32
    observations; povar_create uses sell_max_degree(hp.num_obs))."""
    lib = load()
    sizes = (C.c_int64 * 3)()
    lp = np.ascontiguousarray(hp.lm_ptr, dtype=np.int64)
    oc = np.ascontiguousarray(hp.obs_cam, dtype=np.int32)
    args = (hp.num_cams, hp.num_lms, lp.ctypes.data_as(C.POINTER(C.c_int64)), oc.ctypes.data_as(C.POINTER(C.c_int32)),
            threads, max_deg)
    rc = lib.povar_debug_sell_layout(*args, None, None, None, sizes)
    if rc != OK:
        raise PovarError(rc, "povar_debug_sell_layout failed")
    out = [np.zeros(max(int(n), 1), dtype=np.int32) for n in sizes]
    rc = lib.povar_debug_sell_layout(*args, *[a.ctypes.data_as(C.POINTER(C.c_int32)) for a in out], sizes)
    if rc != OK:
        raise PovarError(rc, "povar_debug_sell_layout failed")
    return tuple(a[:int(n)] for a, n in zip(out, sizes))


def landmark_plan(hp: "HostProblem", model: int = 0, sms: int = 148, max_deg: int = 0):
    """Plan of the landmark half (engine.cu plan_landmark_half) for `hp`: (info dict, range_slice, blk_lo)."""
    lib = load()
    info = (C.c_int64 * 8)()
    lp = np.ascontiguousarray(hp.lm_ptr, dtype=np.int64)
    oc = np.ascontiguousarray(hp.obs_cam, dtype=np.int32)
    args = (hp.num_cams, hp.num_lms, lp.ctypes.data_as(C.POINTER(C.c_int64)), oc.ctypes.data_as(C.POINTER(C.c_int32)),
            model, sms, max_deg, info)
    rc = lib.povar_debug_landmark_plan(*args, None, None)
    if rc != OK:
        raise PovarError(rc, "povar_debug_landmark_plan failed")
    rs = np.zeros(int(info[4]) + 1, dtype=np.int32)
    bl = np.zeros(max(int(info[3]), 1), dtype=np.int32)
    rc = lib.povar_debug_landmark_plan(*args, rs.ctypes.data_as(C.POINTER(C.c_int32)),
                                       bl.ctypes.data_as(C.POINTER(C.c_int32)))
    if rc != OK:
        raise PovarError(rc, "povar_debug_landmark_plan failed")
    names = ("warps", "stages", "blocks_per_sm", "blocks", "ranges", "win_cams", "covered", "smem_bytes")
    return {k: int(v) for k, v in zip(names, info)}, rs, bl[:int(info[3])]


def create_dataset(src: str, dst: str, seed: int = -1) -> None:
    """--create-dataset of the reference (bal_problem.cpp:306-471): BAL file -> 15-parameter file."""
    lib = load()
    err = C.create_string_buffer(512)
    rc = lib.povar_bal_create_dataset(src.encode(), dst.encode(), seed, err, 512)
    if rc != OK:
        raise PovarError(rc, err.value.decode() or "povar_bal_create_dataset failed")


def unique_id() -> bytes:
    lib = load()
    buf = (C.c_uint8 * 128)()
    rc = lib.povar_comm_unique_id(buf)
    if rc != OK:
        raise PovarError(rc, lib.povar_last_error(None).decode())
    return bytes(buf)


def cholesky_solve(A: np.ndarray, b: np.ndarray):
    """x = A^-1 b by the library's own blocked Cholesky (povar_debug_cholesky); returns (x, info)"""
    lib = load()
    A = np.ascontiguousarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    x = np.empty_like(b)
    info = C.c_int32(0)
    rc = lib.povar_debug_cholesky(A.shape[0], _dp(A), _dp(b), _dp(x), C.byref(info))
    if rc != OK:
        raise PovarError(rc, "povar_debug_cholesky failed")
    return x, info.value


def sparse_cholesky_solve(A: np.ndarray, b: np.ndarray, block: int = 12):
    """x = A^-1 b by the library's tile-sparse Cholesky (povar_debug_sparse_cholesky): the pattern is that of the
    non-zero block x block blocks of A's lower triangle.  Returns (x, info, stored_tiles)."""
    lib = load()
    A = np.ascontiguousarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    x = np.empty_like(b)
    info = C.c_int32(0)
    tiles = C.c_int64(0)
    rc = lib.povar_debug_sparse_cholesky(A.shape[0], block, _dp(A), _dp(b), _dp(x), C.byref(info), C.byref(tiles))
    if rc != OK:
        raise PovarError(rc, "povar_debug_sparse_cholesky failed")
    return x, info.value, tiles.value


def cholesky_symbolic(hp: "HostProblem", threads: int = 0):
    """Camera order and stored 64x64 tiles of the tile-sparse CHOLESKY factor of `hp` (povar_debug_cholesky_symbolic):
    (perm, stored_tiles), perm[c] = position of camera c."""
    lib = load()
    lp = np.ascontiguousarray(hp.lm_ptr, dtype=np.int64)
    oc = np.ascontiguousarray(hp.obs_cam, dtype=np.int32)
    perm = np.empty(hp.num_cams, dtype=np.int32)
    tiles = C.c_int64(0)
    rc = lib.povar_debug_cholesky_symbolic(hp.num_cams, hp.num_lms, lp.ctypes.data_as(C.POINTER(C.c_int64)),
                                           oc.ctypes.data_as(C.POINTER(C.c_int32)), threads,
                                           perm.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(tiles))
    if rc != OK:
        raise PovarError(rc, "povar_debug_cholesky_symbolic failed")
    return perm, tiles.value


def host_id() -> bytes:
    """id of a host (shared-memory) rendezvous: no NCCL, ranks may share a device (povar_comm_host_id)"""
    lib = load()
    buf = (C.c_uint8 * 128)()
    rc = lib.povar_comm_host_id(buf)
    if rc != OK:
        raise PovarError(rc, "povar_comm_host_id failed")
    return bytes(buf)


def make_comm(rank: int, world: int, device: int, nccl_id: bytes) -> CommDesc:
    c = CommDesc()
    c.rank, c.world_size, c.device = rank, world, device
    C.memmove(c.nccl_id, nccl_id, 128)
    return c
