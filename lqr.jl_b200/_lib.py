"""ctypes binding of liblqrb200.so (the C ABI in include/lqrb200.h).

There is no fallback: if the shared library is missing, or no sm_100 device is visible when a
handle is requested, this raises.  Nothing under ``oracle/`` is ever imported from here.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LQRB200_LIB", os.path.join(_HERE, "liblqrb200.so"))  # override: kernel A/B experiments only
CSRC = os.path.join(_HERE, "csrc")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "lqrb200.h")

HESS_DENSE, HESS_BLOCKDIAG, HESS_DIAG = 0, 1, 2
FLAG_SOC, FLAG_LTI, FLAG_NO_AFFINE = 1, 2, 4
TILE = 32

_lib = None

c_i32, c_i64, c_vp, c_dp = C.c_int32, C.c_int64, C.c_void_p, C.c_void_p


class LqrbError(RuntimeError):
    pass


class RiccatiLayout(C.Structure):
    _fields_ = [("rows_per_knot", c_i64), ("knot_count", c_i64), ("term_rows", c_i64),
                ("z_rows", c_i64), ("gain_rows", c_i64)]


class SqpOptions(C.Structure):
    _fields_ = [("N", c_i32), ("iters", c_i32), ("dt", C.c_double), ("q_diag", C.c_double),
                ("r_diag", C.c_double), ("qf_diag", C.c_double), ("eps_p", C.c_double),
                ("eps_d", C.c_double), ("line_search", c_i32)]


def build(force: bool = False, jobs: int = 8) -> str:
    """Compile liblqrb200.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    args = ["make", "-C", CSRC, f"-j{jobs}"]
    if force:
        args.append("-B")
    subprocess.run(args, check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


_SIGS = {
    "lqrb_version": (c_i32, []),
    "lqrb_device_count": (c_i32, [C.POINTER(c_i32)]),
    "lqrb_create": (c_i32, [C.POINTER(c_vp), c_i32]),
    "lqrb_destroy": (c_i32, [c_vp]),
    "lqrb_last_error_string": (C.c_char_p, [c_vp]),
    "lqrb_set_stream": (c_i32, [c_vp, c_vp]),
    "lqrb_synchronize": (c_i32, [c_vp]),
    "lqrb_launch_count": (c_i64, [c_vp]),
    "lqrb_last_kernel_name": (C.c_char_p, [c_vp]),
    "lqrb_set_option": (c_i32, [c_vp, C.c_char_p, c_i64]),
    "lqrb_fp64_peak_f64": (c_i32, [c_vp, c_i32, C.c_double, C.POINTER(C.c_double)]),
    "lqrb_padded_batch": (c_i64, [c_i64]),
    "lqrb_num_vars": (c_i64, [c_i32, c_i32, c_i32]),
    "lqrb_num_cons": (c_i64, [c_i32, c_i32, c_vp]),
    "lqrb_riccati_layout": (c_i32, [c_i32, c_i32, c_i32, c_i32, C.POINTER(RiccatiLayout)]),
    "lqrb_kkt_data_rows": (c_i64, [c_i32, c_i32, c_i32, c_vp, c_i32, c_i32]),
    "lqrb_kkt_knot_offset": (c_i64, [c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_i32]),
    "lqrb_riccati_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 12 + [c_vp]),
    "lqrb_riccati_grad_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 19 + [c_vp]),
    "lqrb_riccati_pack_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 11),
    "lqrb_riccati_solve_packed_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 4 + [c_vp]),
    "lqrb_riccati_tile_width": (c_i32, [c_vp, c_i32, c_i32]),
    "lqrb_riccati_unpack_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64] + [c_dp] * 5),
    "lqrb_unpack_rows_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_dp, c_dp]),
    "lqrb_pack_rows_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_dp, c_dp]),
    "lqrb_kkt_tile_width": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32]),
    "lqrb_kkt_unpack_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32] + [c_dp] * 6),
    "lqrb_rollout_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 5),
    "lqrb_lsq_solve_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64] + [c_dp] * 7 + [c_vp]),
    "lqrb_block_cholesky_f64": (c_i32, [c_vp, c_i32, c_i32, c_i64, c_i32] + [c_dp] * 4 + [c_vp]),
    "lqrb_block_ldiv_f64": (c_i32, [c_vp, c_i32, c_i32, c_i64, c_i32, c_dp, c_i32, c_dp]),
    "lqrb_kkt_solve_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32] + [c_dp] * 14 + [c_vp]),
    "lqrb_kkt_pack_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32] + [c_dp] * 12),
    "lqrb_kkt_solve_packed_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32, c_i32]
                                  + [c_dp] * 4 + [c_vp]),
    "lqrb_kkt_factor_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32] + [c_dp] * 7 + [c_vp]),
    "lqrb_kkt_solve_factored_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32, c_i32] + [c_dp] * 7
                                    + [c_vp]),
    "lqrb_kkt_get_shur_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32, c_i32] + [c_dp] * 14 + [c_vp]),
    "lqrb_kkt_last_condition": (c_i32, [c_vp, c_i64, c_vp, C.POINTER(c_i64)]),
    "lqrb_kkt_residual_f64": (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i64, c_vp, c_i32] + [c_dp] * 9),
    "lqrb_sqp_dubins_f64": (c_i32, [c_vp, c_i64, C.POINTER(SqpOptions)] + [c_dp] * 5 + [c_vp, C.POINTER(c_i64)]),
}

EXPORTS = tuple(_SIGS)


def lib() -> C.CDLL:
    """Load the shared library (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LqrbError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def ptr(a):
    """Raw address of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if not a.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        if not a.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return a.data_ptr()
    if isinstance(a, int):
        return a
    raise TypeError(f"cannot take the address of {type(a)}")


class Handle:
    """One lqrb handle = one GPU + one stream (SURVEY §8b threading contract)."""

    def __init__(self, device: int = 0):
        self._h = c_vp()
        L = lib()
        rc = L.lqrb_create(C.byref(self._h), device)
        if rc != 0:
            cnt = c_i32(0)
            L.lqrb_device_count(C.byref(cnt))
            raise LqrbError(f"lqrb_create(device={device}) failed with code {rc} "
                            f"({cnt.value} CUDA device(s) visible; an sm_100 GPU is required, no fallback)")
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().lqrb_destroy(self._h)
            self._h = c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int, what: str):
        if rc != 0:
            msg = lib().lqrb_last_error_string(self._h)
            raise LqrbError(f"{what} failed: code {rc}: {msg.decode() if msg else ''}")

    def call(self, name: str, *args):
        self.check(getattr(lib(), name)(self._h, *args), name)

    def set_stream(self, stream_ptr):
        self.call("lqrb_set_stream", stream_ptr)

    def synchronize(self):
        self.call("lqrb_synchronize")

    def set_option(self, name: str, value: int):
        self.call("lqrb_set_option", name.encode(), int(value))

    @property
    def launches(self) -> int:
        return int(lib().lqrb_launch_count(self._h))

    def kkt_last_condition(self, count: int):
        """(log2 pivot ratios of the last tuned KKT launch, number of instances re-solved by the Cholesky-based kernel)."""
        out = np.zeros(count, dtype=np.int32)
        n = c_i64(0)
        self.call("lqrb_kkt_last_condition", count, out.ctypes.data, C.byref(n))
        return out, int(n.value)

    @property
    def last_kernel(self) -> str:
        return lib().lqrb_last_kernel_name(self._h).decode()


def riccati_layout(n, m, N, flags=0) -> RiccatiLayout:
    out = RiccatiLayout()
    rc = lib().lqrb_riccati_layout(n, m, N, flags, C.byref(out))
    if rc:
        raise LqrbError(f"lqrb_riccati_layout: bad argument {-rc}")
    return out


def padded_batch(batch: int) -> int:
    return int(lib().lqrb_padded_batch(batch))


def _pp(p):
    p = np.ascontiguousarray(p, dtype=np.int32)
    return p, p.ctypes.data


def kkt_data_rows(n, m, N, p, hess_mode, explicit_d2=False) -> int:
    p, pa = _pp(p)
    return int(lib().lqrb_kkt_data_rows(n, m, N, pa, hess_mode, int(explicit_d2)))


def num_vars(n, m, N) -> int:
    return int(lib().lqrb_num_vars(n, m, N))


def num_cons(n, N, p) -> int:
    p, pa = _pp(p)
    return int(lib().lqrb_num_cons(n, N, pa))
