"""ctypes binding of include/gaccum.h -- the only way Python reaches the kernels."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

from . import build as _build

ADAM_WEIGHT_DECAY = 0   # reference optimization.py:107-194
ADAM = 1                # tf.train.AdamOptimizer (02:41, 04:42, another-example.py:135)

OK, EINVAL, ENODEVICE, ECUDA, ENCCL, ENOMEM = 0, -1, -2, -3, -4, -5


class GaccumError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libgaccum error {code}: {msg}")
        self.code = code


class HParams(C.Structure):
    """gaccum_hparams; defaults = what create_optimizer hard-codes (optimization.py:59-65, 84)."""
    _fields_ = [("variant", C.c_int32), ("reserved", C.c_int32), ("beta1", C.c_double),
                ("beta2", C.c_double), ("epsilon", C.c_double), ("weight_decay_rate", C.c_double),
                ("clip_norm", C.c_double)]

    @classmethod
    def bert(cls) -> "HParams":
        return cls(ADAM_WEIGHT_DECAY, 0, 0.9, 0.999, 1e-6, 0.01, 1.0)

    @classmethod
    def tf_adam(cls, beta1=0.9, beta2=0.999, epsilon=1e-8) -> "HParams":
        return cls(ADAM, 0, beta1, beta2, epsilon, 0.0, 0.0)


class StepArgs(C.Structure):
    _fields_ = [("global_step", C.c_int64), ("accum_n", C.c_int32), ("reserved", C.c_int32),
                ("lr", C.c_float), ("beta1_power", C.c_float), ("beta2_power", C.c_float),
                ("reserved2", C.c_float)]


MAX_RANKS = 8
DP_CTRL_BYTES = 256


class DpComm(C.Structure):
    """gaccum_dp_comm: the local accumulator slab + peer base pointers for the fused data-parallel apply."""
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("accum", C.c_void_p),
                ("param_peers", C.c_void_p * MAX_RANKS), ("stage_peers", C.c_void_p * MAX_RANKS),
                ("ctrl_peers", C.c_void_p * MAX_RANKS), ("stage_elements", C.c_int64)]


class DpIpc(C.Structure):
    """gaccum_dp_ipc: what one rank's host session exports for the others (plain bytes)."""
    _fields_ = [("param", C.c_ubyte * 64), ("stage", C.c_ubyte * 64), ("ctrl", C.c_ubyte * 64),
                ("stage_elements", C.c_int64), ("padded_size", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [("applied", C.c_float), ("lr", C.c_float), ("global_norm", C.c_float),
                ("clip_scale", C.c_float)]


_lib = None


def lib_path() -> str:
    _load()                 # make sure it exists (built on demand) before anyone dlopens the path
    return _build.LIB


def _load():
    global _lib
    if _lib is not None:
        return _lib
    try:
        path = _build.build_libgaccum()
    except Exception as e:  # no nvcc and no prebuilt library: fail loudly, never fall back
        if not os.path.exists(_build.LIB):
            raise ImportError(f"libgaccum.so is missing and cannot be built ({e}); "
                              "there is no CPU/PyTorch fallback for the train_op") from e
        path = _build.LIB
    L = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    sig = {
        "gaccum_version": (C.c_int, []),
        "gaccum_last_error": (C.c_char_p, []),
        "gaccum_device_count": (C.c_int, []),
        "gaccum_learning_rate": (C.c_float, [C.c_double, i64, i64, i64]),
        "gaccum_is_apply_step": (C.c_int, [i64, i32]),
        "gaccum_decay_mask": (C.c_int, [i32, vp, C.c_double, vp, i32, vp]),
        "gaccum_plan_create": (C.c_int, [C.POINTER(vp), i32, vp, vp, C.POINTER(HParams), i32]),
        "gaccum_plan_destroy": (C.c_int, [vp]),
        "gaccum_padded_size": (i64, [vp]),
        "gaccum_offsets": (C.c_int, [vp, vp]),
        "gaccum_num_tensors": (i32, [vp]),
        "gaccum_num_elements": (i64, [vp]),
        "gaccum_num_tiles": (i32, [vp]),
        "gaccum_algorithmic_bytes": (i64, [vp, i32]),
        "gaccum_step": (C.c_int, [vp, vp, vp, vp, vp, vp, C.POINTER(StepArgs), vp]),
        "gaccum_accumulate": (C.c_int, [vp, vp, vp, vp]),
        "gaccum_apply": (C.c_int, [vp, vp, vp, vp, vp, vp, C.POINTER(StepArgs), vp]),
        "gaccum_step_packed": (C.c_int, [vp, vp, vp, vp, vp, vp, C.POINTER(StepArgs), i32, vp]),
        "gaccum_read_stats": (C.c_int, [vp, vp, vp]),
        "gaccum_host_session_create": (C.c_int, [C.POINTER(vp), vp]),
        "gaccum_host_session_destroy": (C.c_int, [vp]),
        "gaccum_host_session_set_params": (C.c_int, [vp, vp]),
        "gaccum_step_host": (C.c_int, [vp, vp, vp, C.POINTER(StepArgs), vp]),
        "gaccum_host_session_sync": (C.c_int, [vp]),
        "gaccum_host_session_slabs": (C.c_int, [vp, vp]),
        "gaccum_host_session_dp_export": (C.c_int, [vp, i32, C.POINTER(DpIpc)]),
        "gaccum_host_session_dp_connect": (C.c_int, [vp, i32, i32, C.POINTER(DpIpc)]),
        "gaccum_dp_shard_range": (C.c_int, [vp, i32, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]),
        "gaccum_dp_stage_elements": (i64, [vp, i32]),
        "gaccum_apply_dp": (C.c_int, [vp, C.POINTER(DpComm), vp, vp, vp, C.POINTER(StepArgs), C.c_uint32, vp]),
        "gaccum_step_dp": (C.c_int, [vp, C.POINTER(DpComm), vp, vp, vp, C.POINTER(StepArgs), C.c_uint32, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def _check(rc: int) -> None:
    if rc != 0:
        raise GaccumError(rc, (_load().gaccum_last_error() or b"").decode())


def version() -> int:
    return _load().gaccum_version()


def device_count() -> int:
    return _load().gaccum_device_count()


def learning_rate(init_lr: float, num_train_steps: int, num_warmup_steps: Optional[int], global_step: int) -> float:
    """optimization.py:29-54 in fp32 (host)."""
    return float(_load().gaccum_learning_rate(float(init_lr), int(num_train_steps),
                                              int(num_warmup_steps or 0), int(global_step)))


def is_apply_step(global_step: int, accum_n: int) -> bool:
    """optimization.py:77,91."""
    return bool(_load().gaccum_is_apply_step(int(global_step), int(accum_n)))


def _c_strs(strs: Sequence[str]):
    arr = (C.c_char_p * len(strs))()
    arr[:] = [s.encode() for s in strs]
    return arr


def decay_mask(names: Sequence[str], weight_decay_rate: float,
               exclude: Optional[Sequence[str]] = ("LayerNorm", "layer_norm", "bias")) -> List[bool]:
    """optimization.py:179-194, with the reference's own regular-expression engine: Python ``re.search`` on the
    name with a trailing ``:<digits>`` stripped.  (The C helper ``gaccum_decay_mask`` is for non-Python callers and
    speaks POSIX ERE: identical for the reference's plain substrings, different for Python-only syntax such as
    ``\\d`` or look-arounds -- both Python bindings therefore evaluate the patterns here.)"""
    import re
    out = []
    for n in names:
        m = re.match("^(.*):\\d+$", n)                      # _get_variable_name, optimization.py:189-194
        if m is not None:
            n = m.group(1)
        use = bool(weight_decay_rate)                       # :181
        if use and exclude:
            for r in exclude:
                if re.search(r, n) is not None:             # :183-186
                    use = False
        out.append(use)
    return out


def decay_mask_c(names: Sequence[str], weight_decay_rate: float,
                 exclude: Optional[Sequence[str]] = ("LayerNorm", "layer_norm", "bias")) -> List[bool]:
    """The C ABI's ``gaccum_decay_mask`` (POSIX extended regular expressions)."""
    exclude = list(exclude or [])
    out = (C.c_uint8 * len(names))()
    n, e = _c_strs(names), _c_strs(exclude)
    _check(_load().gaccum_decay_mask(len(names), C.cast(n, C.c_void_p), float(weight_decay_rate),
                                     C.cast(e, C.c_void_p), len(exclude), C.cast(out, C.c_void_p)))
    return [bool(x) for x in out]


class Plan:
    """gaccum_plan: slab layout + tile table for T tensors.  device=-1 -> layout-only."""

    def __init__(self, numels: Sequence[int], decay: Optional[Sequence[bool]], hp: HParams, device: int = -1):
        L = _load()
        self.T = len(numels)
        self.hp = hp
        self.device = device
        ne = (C.c_int64 * self.T)(*[int(n) for n in numels])
        dm = (C.c_uint8 * self.T)(*[1 if d else 0 for d in (decay or [0] * self.T)])
        h = C.c_void_p()
        _check(L.gaccum_plan_create(C.byref(h), self.T, C.cast(ne, C.c_void_p), C.cast(dm, C.c_void_p),
                                    C.byref(hp), int(device)))
        self._h = h
        self.numels = [int(n) for n in numels]
        self.padded_size = int(L.gaccum_padded_size(h))
        self.num_elements = int(L.gaccum_num_elements(h))
        self.num_tiles = int(L.gaccum_num_tiles(h))
        off = (C.c_int64 * self.T)()
        _check(L.gaccum_offsets(h, C.cast(off, C.c_void_p)))
        self.offsets = [int(x) for x in off]

    def algorithmic_bytes(self, is_apply: bool) -> int:
        return int(_load().gaccum_algorithmic_bytes(self._h, 1 if is_apply else 0))

    @staticmethod
    def ptr_array(ptrs: Sequence[int]):
        return (C.c_void_p * len(ptrs))(*[p if p else None for p in ptrs])

    def step(self, grads, params, accum: int, m: int, v: int, args: StepArgs, stream: int = 0) -> None:
        _check(_load().gaccum_step(self._h, grads, params, accum, m, v, C.byref(args), stream))

    def accumulate(self, grads, accum: int, stream: int = 0) -> None:
        _check(_load().gaccum_accumulate(self._h, grads, accum, stream))

    def apply(self, grads, params, accum: int, m: int, v: int, args: StepArgs, stream: int = 0) -> None:
        _check(_load().gaccum_apply(self._h, grads, params, accum, m, v, C.byref(args), stream))

    def step_packed(self, grad_slab: int, param_slab: int, accum: int, m: int, v: int, args: StepArgs,
                    force_branch: int = -1, stream: int = 0) -> None:
        _check(_load().gaccum_step_packed(self._h, grad_slab or None, param_slab or None, accum, m, v,
                                          C.byref(args), force_branch, stream))

    def dp_shard_range(self, world: int, rank: int):
        lo, hi, n = C.c_int32(), C.c_int32(), C.c_int64()
        _check(_load().gaccum_dp_shard_range(self._h, world, rank, C.byref(lo), C.byref(hi), C.byref(n)))
        return lo.value, hi.value, n.value

    def dp_stage_elements(self, world: int) -> int:
        n = int(_load().gaccum_dp_stage_elements(self._h, world))
        if n < 0:
            _check(n)
        return n

    def apply_dp(self, comm: "DpComm", grads, m: int, v: int, args: StepArgs, epoch: int, stream: int = 0) -> None:
        _check(_load().gaccum_apply_dp(self._h, C.byref(comm), grads, m, v, C.byref(args), epoch, stream))

    def step_dp(self, comm: "DpComm", grads, m: int, v: int, args: StepArgs, epoch: int, stream: int = 0) -> None:
        _check(_load().gaccum_step_dp(self._h, C.byref(comm), grads, m, v, C.byref(args), epoch, stream))

    def read_stats(self, host_ptr: int, stream: int = 0) -> None:
        _check(_load().gaccum_read_stats(self._h, host_ptr, stream))

    def close(self) -> None:
        if getattr(self, "_h", None):
            _load().gaccum_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostSession:
    """gaccum_host_session: the train_op for a caller whose tensors live in host memory."""

    def __init__(self, plan: Plan):
        self.plan = plan
        h = C.c_void_p()
        _check(_load().gaccum_host_session_create(C.byref(h), plan._h))
        self._h = h

    def set_params(self, host_ptrs) -> None:
        _check(_load().gaccum_host_session_set_params(self._h, host_ptrs))

    def step(self, host_grad_ptrs, host_param_out_ptrs, args: StepArgs, stats_ptr: int = 0) -> None:
        _check(_load().gaccum_step_host(self._h, host_grad_ptrs, host_param_out_ptrs, C.byref(args), stats_ptr or None))

    def sync(self) -> None:
        _check(_load().gaccum_host_session_sync(self._h))

    def dp_export(self, world: int) -> bytes:
        rec = DpIpc()
        _check(_load().gaccum_host_session_dp_export(self._h, world, C.byref(rec)))
        return bytes(rec)

    def dp_connect(self, rank: int, world: int, records: Sequence[bytes]) -> None:
        arr = (DpIpc * world)()
        for w, r in enumerate(records):
            C.memmove(C.byref(arr[w]), r, C.sizeof(DpIpc))
        _check(_load().gaccum_host_session_dp_connect(self._h, rank, world, arr))

    def slabs(self):
        out = (C.c_void_p * 4)()
        _check(_load().gaccum_host_session_slabs(self._h, out))
        return [int(x) for x in out]

    def close(self) -> None:
        if getattr(self, "_h", None):
            _load().gaccum_host_session_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
