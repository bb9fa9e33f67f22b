"""ctypes binding of libtwisterl_b200.so (the C ABI in include/twisterl_b200.h).

There is no CPU fallback: if the CUDA library cannot be loaded, or no B200-class device is
present when an engine is needed, every product entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "lib" / "libtwisterl_b200.so"

OK = 0
ENV_PUZZLE, ENV_GRIDWORLD = 0, 1
ABI_VERSION = 3                      # TWR_ABI_VERSION of the header these struct layouts / prototypes were written against
PREC_FP32, PREC_F16X2, PREC_F16X2_W16, PREC_F16_F8C = 0, 1, 2, 3
PRECISIONS = {"fp32": PREC_FP32, "f16x2": PREC_F16X2, "f16x2w16": PREC_F16X2_W16, "f16f8c": PREC_F16_F8C}
# the tcgen05 forward: all operands split / common-layer weight as one fp16 term / that with the correction products in fp8
TC_PRECISIONS = ("f16x2", "f16x2w16", "f16f8c")
MAX_ACTIONS = 4

f32p, i32p, i64p, u8p, i8p, u16p = (C.POINTER(t) for t in (C.c_float, C.c_int32, C.c_int64, C.c_uint8, C.c_int8, C.c_uint16))


class EngineCfg(C.Structure):
    _fields_ = [("device", C.c_int32), ("precision", C.c_int32), ("seed", C.c_uint64),
                ("rank", C.c_int32), ("world", C.c_int32), ("stream", C.c_void_p)]


class EnvSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                ("difficulty", C.c_int32), ("depth_slope", C.c_int32), ("max_depth", C.c_int32)]


class LinearDesc(C.Structure):
    _fields_ = [("weights", f32p), ("bias", f32p), ("in_", C.c_int32), ("out", C.c_int32), ("apply_relu", C.c_int32)]


class PolicyDesc(C.Structure):
    _fields_ = [("emb_vectors", f32p), ("emb_bias", f32p), ("obs_size", C.c_int32), ("emb_size", C.c_int32),
                ("emb_apply_relu", C.c_int32), ("obs_shape", C.c_int32 * 2), ("obs_shape_len", C.c_int32),
                ("conv_dim", C.c_int32),
                ("common", C.POINTER(LinearDesc)), ("n_common", C.c_int32),
                ("action_net", C.POINTER(LinearDesc)), ("n_action", C.c_int32),
                ("value_net", C.POINTER(LinearDesc)), ("n_value", C.c_int32),
                ("obs_perms", i32p), ("act_perms", i32p), ("n_perms", C.c_int32)]


class Collected(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("num_episodes", C.c_int64), ("n_cells", C.c_int32),
                ("num_actions", C.c_int32), ("successes", C.c_int64), ("reward_sum", C.c_double),
                ("obs", C.c_void_p), ("logits", C.c_void_p), ("values", C.c_void_p), ("rewards", C.c_void_p),
                ("advs", C.c_void_p), ("rets", C.c_void_p), ("actions", C.c_void_p), ("perms", C.c_void_p),
                ("ep_len", C.c_void_p)]


class HostBuffers(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("obs", C.c_void_p), ("logits", C.c_void_p), ("values", C.c_void_p),
                ("rewards", C.c_void_p), ("advs", C.c_void_p), ("rets", C.c_void_p), ("actions", C.c_void_p),
                ("perms", C.c_void_p), ("ep_len", C.c_void_p), ("obs_u8", C.c_void_p)]


# every symbol include/twisterl_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "twr_abi_version", "twr_last_error", "twr_device_count", "twr_engine_create", "twr_engine_destroy",
    "twr_engine_synchronize", "twr_engine_launch_count", "twr_policy_create", "twr_policy_update",
    "twr_policy_create_from_safetensors", "twr_policy_blob_floats", "twr_policy_update_from_device", "twr_policy_blob_device_ptr", "twr_policy_destroy",
    "twr_envs_create", "twr_envs_destroy", "twr_envs_set_difficulty", "twr_envs_set_state", "twr_envs_set_cell", "twr_envs_reset",
    "twr_envs_step", "twr_envs_get_state", "twr_envs_observe", "twr_envs_masks", "twr_envs_reward",
    "twr_envs_is_final", "twr_envs_success", "twr_envs_depth", "twr_policy_forward", "twr_policy_forward_obs", "twr_policy_full_predict", "twr_debug_forward_profile", "twr_debug_set_tc_terms", "twr_sample", "twr_gae",
    "twr_ppo_collect", "twr_engine_set_collect_id", "twr_collected_to_host", "twr_max_records",
    "twr_ppo_collect_host", "twr_evaluate", "twr_evaluate_episodes", "twr_solve", "twr_az_collect", "twr_mcts_probs", "twr_debug_mcts_trace", "twr_comm_version", "twr_comm_unique_id", "twr_comm_init", "twr_comm_destroy", "twr_broadcast_weights", "twr_allreduce_stats", "twr_gather_collected",
    "twr_host_alloc", "twr_host_free", "twr_engine_set_timing", "twr_engine_last_timing",
]

_lib = None
_lock = threading.Lock()


def load():
    """Load (building it first if it is missing or stale) the CUDA library.  Raises on failure."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        from . import build as _build
        try:
            if _build.is_stale():
                _build.build()
        except Exception as exc:  # nvcc missing etc.
            if not LIB_PATH.exists():
                raise ImportError(f"twisterl_b200: CUDA library missing and cannot be built: {exc}") from exc
            import warnings
            warnings.warn(f"twisterl_b200: sources are newer than {LIB_PATH.name} and the rebuild failed ({exc}); "
                          "loading the existing library (its ABI version is checked)", RuntimeWarning)
        path = os.environ.get("TWISTERL_B200_LIB") or str(LIB_PATH)      # a specific build (A/B runs of kernel variants)
        try:
            L = C.CDLL(path)
        except OSError as exc:
            raise ImportError(f"twisterl_b200: cannot load {path}: {exc} (there is no CPU fallback)") from exc
        if int(L.twr_abi_version()) != ABI_VERSION:
            raise ImportError(f"twisterl_b200: {LIB_PATH} has ABI version {int(L.twr_abi_version())}, this package binds "
                              f"version {ABI_VERSION}: rebuild with `python -m twisterl_b200.build --force`")
        vp = C.c_void_p
        L.twr_last_error.restype = C.c_char_p
        L.twr_engine_create.argtypes = [C.POINTER(EngineCfg), C.POINTER(vp)]
        L.twr_engine_destroy.argtypes = [vp]; L.twr_engine_destroy.restype = None
        L.twr_engine_synchronize.argtypes = [vp]
        L.twr_engine_launch_count.argtypes = [vp]; L.twr_engine_launch_count.restype = C.c_int64
        L.twr_engine_set_collect_id.argtypes = [vp, C.c_uint32]
        L.twr_engine_set_timing.argtypes = [vp, C.c_int32]
        L.twr_engine_last_timing.argtypes = [vp, f32p, f32p, i64p]
        L.twr_policy_create.argtypes = [vp, C.POINTER(PolicyDesc), C.POINTER(vp)]
        L.twr_policy_update.argtypes = [vp, C.POINTER(PolicyDesc)]
        L.twr_policy_create_from_safetensors.argtypes = [vp, C.c_char_p, i32p, C.c_int32, C.c_int32, i32p, i32p, C.c_int32, C.POINTER(vp)]
        L.twr_policy_blob_floats.argtypes = [vp]; L.twr_policy_blob_floats.restype = C.c_int64
        L.twr_policy_update_from_device.argtypes = [vp, vp]
        L.twr_policy_blob_device_ptr.argtypes = [vp, C.POINTER(vp)]
        L.twr_policy_destroy.argtypes = [vp]; L.twr_policy_destroy.restype = None
        L.twr_envs_create.argtypes = [vp, C.POINTER(EnvSpec), C.c_int64, C.POINTER(vp)]
        L.twr_envs_destroy.argtypes = [vp]; L.twr_envs_destroy.restype = None
        L.twr_envs_set_difficulty.argtypes = [vp, C.c_int32]
        L.twr_envs_set_state.argtypes = [vp, vp]
        L.twr_envs_set_cell.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32]
        L.twr_envs_reset.argtypes = [vp, C.c_uint32, C.c_uint32]
        for name in ("step", "get_state", "observe", "masks", "reward", "is_final", "success", "depth"):
            getattr(L, "twr_envs_" + name).argtypes = [vp, vp]
        L.twr_policy_forward.argtypes = [vp, vp, vp, vp, C.c_int32, vp, vp]
        L.twr_policy_forward_obs.argtypes = [vp, vp, vp, C.c_int64, C.c_int32, vp, vp, vp]
        L.twr_policy_full_predict.argtypes = [vp, vp, vp, vp, vp]
        L.twr_debug_forward_profile.argtypes = [vp, vp, vp, vp, C.c_int32, C.c_int32]
        L.twr_debug_set_tc_terms.argtypes = [vp, C.c_int32]
        L.twr_sample.argtypes = [vp, vp, C.c_int64, C.c_int32, C.c_uint32, C.c_uint32, C.c_uint32, vp, vp]
        L.twr_gae.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_float, C.c_float, vp, vp]
        L.twr_ppo_collect.argtypes = [vp, C.POINTER(EnvSpec), vp, C.c_int64, C.c_float, C.c_float, C.POINTER(Collected)]
        L.twr_collected_to_host.argtypes = [vp, C.POINTER(HostBuffers)]
        L.twr_max_records.argtypes = [C.POINTER(EnvSpec), C.c_int64]; L.twr_max_records.restype = C.c_int64
        L.twr_ppo_collect_host.argtypes = [vp, C.POINTER(EnvSpec), vp, C.POINTER(PolicyDesc), C.c_int64, C.c_float,
                                           C.c_float, C.POINTER(HostBuffers), C.POINTER(Collected)]
        L.twr_evaluate.argtypes = [vp, C.POINTER(EnvSpec), vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                   f32p, f32p]
        L.twr_evaluate_episodes.argtypes = [vp, C.POINTER(EnvSpec), vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32,
                                            f32p, f32p, vp, vp]
        L.twr_solve.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32, f32p, f32p, vp, C.c_int32, i32p]
        L.twr_az_collect.argtypes = [vp, C.POINTER(EnvSpec), vp, C.c_int64, C.c_int32, C.c_float, C.c_int32, C.POINTER(Collected)]
        L.twr_mcts_probs.argtypes = [vp, vp, vp, C.c_int32, C.c_float, C.c_int32, C.c_uint32, C.c_uint32, C.c_int32, vp, vp]
        L.twr_comm_unique_id.argtypes = [vp]
        L.twr_comm_init.argtypes = [vp, vp]
        L.twr_comm_destroy.argtypes = [vp]; L.twr_comm_destroy.restype = None
        L.twr_broadcast_weights.argtypes = [vp, vp, C.c_int32]
        L.twr_allreduce_stats.argtypes = [vp, vp, C.c_int32, C.c_int32]
        L.twr_gather_collected.argtypes = [vp, C.c_int32, C.POINTER(Collected)]
        L.twr_debug_mcts_trace.argtypes = [vp, vp, vp, C.c_int32, C.c_float, C.c_int32, C.c_uint32, C.c_uint32, C.c_int32, vp, vp, vp]
        L.twr_host_alloc.argtypes = [C.POINTER(vp), C.c_int64]
        L.twr_host_free.argtypes = [vp]; L.twr_host_free.restype = None
        _lib = L
        return L


def check(rc: int) -> None:
    """Non-zero status -> RuntimeError(message), the mapping of python_interface/error_mapping.rs:29-33."""
    if rc != OK:
        msg = load().twr_last_error()
        raise RuntimeError((msg or b"twisterl_b200 error").decode("utf-8", "replace"))


def ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


# --------------------------------------------------------------------------- engine ---
class Engine:
    """One engine per CUDA device (twr_engine)."""

    def __init__(self, device: int = 0, precision: str | int = "f16x2", seed: int = 0x5EED5EED, rank: int = 0,
                 world: int = 1, stream: int | None = None):
        L = load()
        prec = PRECISIONS[precision] if isinstance(precision, str) else int(precision)
        cfg = EngineCfg(int(device), prec, int(seed) & 0xFFFFFFFFFFFFFFFF, int(rank), int(world), stream)
        h = C.c_void_p()
        check(L.twr_engine_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.device, self.precision, self.seed, self.rank, self.world = int(device), prec, int(seed), int(rank), int(world)

    @property
    def precision_name(self) -> str:
        return {v: k for k, v in PRECISIONS.items()}[self.precision]

    def close(self):
        if getattr(self, "_h", None):
            load().twr_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self): check(load().twr_engine_synchronize(self._h))
    def launch_count(self) -> int: return int(load().twr_engine_launch_count(self._h))
    def set_collect_id(self, cid: int): check(load().twr_engine_set_collect_id(self._h, int(cid)))
    def set_timing(self, on: bool): check(load().twr_engine_set_timing(self._h, int(bool(on))))

    def set_tc_terms(self, terms: int):
        """Debug / precision ladder: split-operand terms of the tensor-core forward (see twr_debug_set_tc_terms)."""
        check(load().twr_debug_set_tc_terms(self._h, int(terms)))

    def last_timing(self):
        f, t, n = C.c_float(), C.c_float(), C.c_int64()
        check(load().twr_engine_last_timing(self._h, C.byref(f), C.byref(t), C.byref(n)))
        return float(f.value), float(t.value), int(n.value)


_default_engine: Engine | None = None
_default_cfg: dict = {}


def configure(**kw) -> None:
    """Set the parameters of the process-wide default engine (device, precision, seed, rank, world).
    Env vars TWISTERL_B200_DEVICE / _PRECISION / _SEED provide defaults."""
    global _default_engine
    _default_cfg.update(kw)
    if _default_engine is not None:
        _default_engine.close()
        _default_engine = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        cfg = dict(device=int(os.environ.get("TWISTERL_B200_DEVICE", os.environ.get("LOCAL_RANK", "0"))),
                   precision=os.environ.get("TWISTERL_B200_PRECISION", "f16x2"),
                   seed=int(os.environ.get("TWISTERL_B200_SEED", str(0x5EED5EED)), 0))
        cfg.update(_default_cfg)
        _default_engine = Engine(**cfg)
    return _default_engine


class PinnedArray:
    """numpy view over cudaHostAlloc'ed memory (twr_host_alloc) for the e2e D2H path."""

    def __init__(self, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(load().twr_host_alloc(C.byref(p), nbytes))
        self._p = p
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def __del__(self):
        try:                                   # at interpreter shutdown the module globals may already be gone
            if getattr(self, "_p", None):
                self.array = None
                load().twr_host_free(self._p)
                self._p = None
        except Exception:
            pass
