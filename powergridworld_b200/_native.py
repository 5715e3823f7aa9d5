"""ctypes binding of the C ABI declared in include/pgw.h (libpgw_b200.so).

There is no CPU fallback: if the shared library is missing the import of the
package still works (so that spaces/configs can be inspected), but creating an
env raises.  The library itself refuses devices that are not sm_100.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PGW_B200_LIB: an instrumented build of the same library (tools/phase_probe.py)
LIB_PATH = os.environ.get("PGW_B200_LIB") or os.path.join(_HERE, "libpgw_b200.so")

ABI_VERSION = 1
NUM_STATS = 8

STORAGE, PV, EV, BUILDING = 1, 2, 3, 4
HS_BEGIN, HS_PV, HS_STORAGE, HS_EV, HS_DEVICES = 5, 6, 7, 8, 9
HS_MAX_COMPONENTS = 8
F_TELEMETRY, HS_TEL_ROWS = 32, 13
F_RESCALE, F_GRID_AWARE, F_PV_VOLT_REWARD, F_STALE_REWARD, F_BUILDING_FAST = 1, 2, 4, 8, 16
F_EV_PER_ENV = 64

OPT_PF_KERNEL, OPT_WARM_START, OPT_GRAPHS, OPT_PDL, OPT_CLIP_INIT_SOC = 0, 1, 2, 3, 4
OPT_PF_POLISH, OPT_PF_TC_TOL_NANO, OPT_FUSED, OPT_HOST_CHUNKS, OPT_HOST_ZERO_COPY = 5, 6, 7, 8, 9

(FIELD_STATE_D, FIELD_STATE_I, FIELD_AGENT_P, FIELD_VOLTAGES, FIELD_VMIN, FIELD_VMAX,
 FIELD_VBUS, FIELD_PF_ITERS, FIELD_EP_RETURN, FIELD_PF_STATE) = range(10)


class Component(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "type", "agent", "flags", "act_off", "obs_off", "obs_dim", "sd_off", "si_off",
        "dtab_off", "itab_off", "dpar_off", "ipar_off")]


class Agent(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("comp_begin", "comp_end", "load_slot", "bus_node")]


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class Feeder(C.Structure):
    _fields_ = [
        ("nb", C.c_int32), ("nn", C.c_int32), ("nl", C.c_int32), ("max_iter", C.c_int32),
        ("tol", C.c_double),
        ("zbb", _dp), ("u0", _dp), ("znb", _dp), ("w", _dp),
        ("branch_load", _ip), ("branch_share", _dp), ("branch_model", _ip),
        ("vminpu", _dp), ("vmaxpu", _dp),
        ("penalty_node", C.c_int32),
        ("penalty_vlo", C.c_double), ("penalty_vhi", C.c_double), ("penalty_unit", C.c_double),
    ]


class Spec(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "abi_version", "num_envs", "num_agents", "num_components", "act_dim", "obs_dim",
        "sd_rows", "si_rows", "num_storage", "num_events", "dtab_stride", "itab_stride",
        "dpar_len", "ipar_len")] + [
        ("agents", C.POINTER(Agent)), ("components", C.POINTER(Component)),
        ("dpar", _dp), ("ipar", _ip), ("dtab", _dp), ("itab", _ip),
        ("feeder", C.POINTER(Feeder)),
    ]


# every symbol include/pgw.h declares: (name, restype, argtypes)
_vp = C.c_void_p
SYMBOLS = {
    "pgw_create": (C.c_int, [C.POINTER(Spec), C.POINTER(_vp)]),
    "pgw_destroy": (C.c_int, [_vp]),
    "pgw_reset": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pgw_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "pgw_reset_host": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pgw_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "pgw_get": (C.c_int, [_vp, C.c_int, _vp, C.c_size_t, _vp]),
    "pgw_set": (C.c_int, [_vp, C.c_int, _vp, C.c_size_t, _vp]),
    "pgw_set_rows": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_size_t, _vp]),
    "pgw_set_clock": (C.c_int, [_vp, C.c_int, _vp]),
    "pgw_update_tables": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp]),
    "pgw_stats": (C.c_int, [_vp, _vp, _vp]),
    "pgw_clock": (C.c_int, [_vp]),
    "pgw_launch_count": (C.c_longlong, [_vp]),
    "pgw_graph_captures": (C.c_longlong, [_vp]),
    "pgw_reset_count": (C.c_longlong, [_vp]),
    "pgw_set_reset_count": (C.c_int, [_vp, C.c_longlong]),
    "pgw_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "pgw_pf_solve": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pgw_set_timing": (C.c_int, [_vp, C.c_int]),
    "pgw_get_timing": (C.c_int, [_vp, _vp, _vp]),
    "pgw_last_error": (C.c_char_p, []),
    "pgw_abi_version": (C.c_int, []),
}

# the float32 I/O forms of reset / step (include/pgw.h, names ending in _f32).  Kept apart from SYMBOLS on
# purpose: tests/test_abi.py checks SYMBOLS against the declarations it parses from pgw.h with the pattern
# pgw_[a-z_]+, which does not match names with digits; tests/test_io_f32_cpu.py checks this table.
# lib() binds both.
SYMBOLS_F32 = {
    "pgw_reset_f32": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pgw_step_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "pgw_reset_host_f32": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pgw_step_host_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Load libpgw_b200.so (built by __graft_entry__.build() / csrc/build.sh)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} is missing: build it with powergridworld_b200/csrc/build.sh "
                "(there is no CPU fallback)")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in {**SYMBOLS, **SYMBOLS_F32}.items():
            fn = getattr(h, name)          # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        if h.pgw_abi_version() != ABI_VERSION:
            raise NativeError("libpgw_b200.so ABI version mismatch")
        _lib = h
    return _lib


def check(rc: int):
    if rc != 0:
        msg = lib().pgw_last_error()
        raise NativeError(f"pgw error {rc}: {msg.decode() if msg else ''}")
