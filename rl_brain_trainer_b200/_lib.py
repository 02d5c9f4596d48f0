"""Loader of ``libkin_b200.so`` (the C ABI in ``include/kin_b200.h``) and ctypes views of its structs.

There is deliberately no fallback: if the library has not been built (``__graft_entry__.build()`` /
``python -m rl_brain_trainer_b200.build``) or cannot be loaded, :func:`lib` raises.
"""

from __future__ import annotations

import ctypes
import re
from pathlib import Path
from typing import Any

PKG_DIR = Path(__file__).resolve().parent
REPO_ROOT = PKG_DIR.parent
HEADER = REPO_ROOT / "include" / "kin_b200.h"
import os

# KIN_B200_LIB: load another build of the same C ABI (experiment / trace builds under tools/_bin); default = the in-tree library
LIB_PATH = Path(os.environ["KIN_B200_LIB"]).resolve() if os.environ.get("KIN_B200_LIB") else PKG_DIR / "libkin_b200.so"

_SCALARS = {"float": ctypes.c_float, "int": ctypes.c_int, "double": ctypes.c_double, "uint32_t": ctypes.c_uint32, "uint64_t": ctypes.c_uint64}
_structs: dict[str, type] = {}
_defines: dict[str, int] = {}


def _header_text() -> str:
    return HEADER.read_text()


def c_struct(name: str) -> type:
    """ctypes.Structure for ``typedef struct <name> {...} <name>;`` parsed from the header."""
    if name in _structs:
        return _structs[name]
    m = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), _header_text(), re.S)
    if m is None:
        raise RuntimeError(f"struct {name} not found in {HEADER}")
    body = re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S)
    fields: list[tuple[str, Any]] = []
    for raw in body.split(";"):
        line = raw.strip()
        if not line:
            continue
        mm = re.match(r"(const\s+)?(\w+)\s*(\*)?\s*(\w+)(?:\[(\d+)\])?$", line)
        if mm is None:
            raise RuntimeError(f"cannot parse field {line!r} of {name}")
        _, ctype, ptr, fname, arr = mm.groups()
        t: Any = ctypes.c_void_p if ptr else (_SCALARS[ctype] if ctype in _SCALARS else c_struct(ctype))      # (a nested Kin* struct)
        if arr:
            t = t * int(arr)
        fields.append((fname, t))
    cls = type(name, (ctypes.Structure,), {"_fields_": fields})
    _structs[name] = cls
    return cls


def define(name: str) -> int:
    """Integer value of a ``#define KIN_*`` constant in the header."""
    if not _defines:
        for m in re.finditer(r"^#define\s+(KIN_\w+)\s+\(?(-?(?:0x[0-9a-fA-F]+|\d+))u?\)?", _header_text(), re.M):
            _defines[m.group(1)] = int(m.group(2), 0)
    return _defines[name]


def declared_functions() -> list[str]:
    """Names of every function the header declares (used by the CPU-side symbol test)."""
    text = re.sub(r"/\*.*?\*/", "", _header_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(kin_\w+)\s*\(", text)))


_lib: ctypes.CDLL | None = None


class KinError(RuntimeError):
    """A C-ABI call returned a non-zero code (message from kin_last_error_string)."""


def library_source_hash(path: Path | None = None) -> str:
    """``kin_source_hash()`` of a built library, read through a throw-away handle (``"missing"`` if the symbol is absent)."""
    h = ctypes.CDLL(str(path or LIB_PATH))
    try:
        fn = h.kin_source_hash
    except AttributeError:
        return "missing"
    fn.restype = ctypes.c_char_p
    return fn().decode()


def _check_source_hash() -> None:
    """The in-tree library must have been compiled from the sources it sits next to (``build.source_hash``).  A stale library is
    rebuilt once when nvcc is there (the GPU box has the same image); otherwise, or if the rebuild does not fix it, loading fails.
    ``KIN_B200_ALLOW_STALE=1`` turns the refusal into a warning (experiments with hand-built libraries)."""
    from . import build as kbuild

    want = kbuild.source_hash()
    got = library_source_hash()
    if got == want:
        return
    if os.environ.get("KIN_B200_ALLOW_STALE"):
        import warnings

        warnings.warn(f"libkin_b200.so was built from other sources (library {got[:12]}, tree {want[:12]})")
        return
    try:
        kbuild.build()
    except Exception as exc:  # no nvcc, compile error ...
        raise KinError(f"libkin_b200.so was built from other sources (library {got[:12]}, tree {want[:12]}) and the rebuild failed: {exc}") from exc
    got = library_source_hash()
    if got != want:
        raise KinError(f"libkin_b200.so does not match its sources after a rebuild (library {got[:12]}, tree {want[:12]})")


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise KinError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(nvcc, sm_100a). There is no CPU fallback.")
    default_lib = not os.environ.get("KIN_B200_LIB") and LIB_PATH == PKG_DIR / "libkin_b200.so"
    if default_lib:
        _check_source_hash()
    L = ctypes.CDLL(str(LIB_PATH))
    vp, i32, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64
    L.kin_abi_version.restype = i32
    L.kin_last_error_string.restype = ctypes.c_char_p
    L.kin_device_info.argtypes = [ctypes.POINTER(i32)] * 3 + [ctypes.c_char_p, i32]
    L.kin_params_create.argtypes = [vp, ctypes.POINTER(vp)]
    L.kin_params_set_sampler.argtypes = [vp, vp]
    L.kin_params_destroy.argtypes = [vp]
    L.kin_fk_pose6.argtypes = [vp, vp, vp, i32, vp]
    L.kin_env_reset.argtypes = [vp, vp, i32, i32, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp]
    L.kin_env_reset_sampled.argtypes = [vp, vp, i32, i32, vp, i32, u64, vp, vp]
    L.kin_env_step.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, u64, vp, vp]
    L.kin_env_observe.argtypes = [vp, vp, i32, i32, vp, vp]
    L.kin_policy_forward.argtypes = [vp, vp, vp, vp, i32, vp]
    L.kin_rollout_approach_finisher.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]
    L.kin_rollout_handoff_states.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]
    L.kin_route_reset.argtypes = [vp, vp, vp, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.kin_route_reset_sampled.argtypes = [vp, vp, vp, vp, i32, i32, vp, u64, ctypes.c_uint32, vp, vp]
    L.kin_route_step.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    L.kin_route_step_autoreset.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, i32, i32, u64, vp, vp]
    L.kin_route_probe.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]
    L.kin_route_probe_rows.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, vp]
    L.kin_route_probe_tc.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp]
    f32, i64, u32 = ctypes.c_float, ctypes.c_longlong, ctypes.c_uint32
    L.kin_ppo_param_count.argtypes = [i32]
    L.kin_policy_act.argtypes = [vp, vp, vp, vp, vp, i32, u64, u32, i32, vp]
    L.kin_ppo_bootstrap.argtypes = [vp, vp, vp, vp, f32, i32, vp]
    L.kin_ppo_gae.argtypes = [vp, vp, vp, vp, vp, f32, f32, i32, i32, vp, vp, vp, vp]
    L.kin_ppo_grad.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp, i32, vp, vp, vp, vp]
    L.kin_ppo_adam.argtypes = [vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, i32, vp]
    L.kin_ppo_pack_weights.argtypes = [vp, i32, vp, vp]
    L.kin_ppo_grad_tc.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp, i32, vp, vp, vp, vp, i32, i32, vp, vp, vp]
    L.kin_ppo_grad_tc_exchange.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp, i32, vp, vp, i32, vp, vp, vp, i32, i32, u32, vp, vp]
    L.kin_ppo_tc3_config.argtypes = [i32, i32]
    L.kin_ppo_grad_tc_update.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, vp, i32, vp, vp, i32, vp, vp, vp, i32, i32, u32, vp, vp, vp, vp, i32, vp, vp, vp]
    L.kin_ppo_shuffle.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.kin_ppo_adv_stats.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    L.kin_ppo_collect.argtypes = [vp, vp, i32, i32, i32, vp, vp, i32, i32, u64, u32, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    L.kin_ppo_bootstrap_list.argtypes = [vp, i32, vp, vp, vp, i32, vp, f32, vp]
    L.kin_route_obs_images.argtypes = [vp, i64, vp, vp]
    L.kin_route_collect.argtypes = [vp, vp, vp, vp, i32, i32, vp, i32, u64, u32, u64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    L.kin_params_device_sampler.argtypes = [vp, ctypes.POINTER(vp)]
    L.kin_params_same_env.argtypes = [vp, vp, ctypes.POINTER(i32)]
    L.kin_pop_collect.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    L.kin_pop_bootstrap_list.argtypes = [vp, i32, i32, vp]
    L.kin_pop_gae.argtypes = [vp, i32, i32, i32, vp]
    L.kin_pop_adv_stats.argtypes = [vp, i32, i32, i32, vp]
    L.kin_pop_grad_tc.argtypes = [vp, i32, i32, i32, i64, i32, vp]
    L.kin_pop_adam.argtypes = [vp, i32, vp, vp, vp]
    L.kin_peer_buffer_bytes.argtypes = [i32, i32]
    L.kin_peer_buffer_create.argtypes = [i32, i32, ctypes.POINTER(vp), ctypes.c_char_p]
    L.kin_peer_buffer_open.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
    L.kin_peer_buffer_close.argtypes = [vp]
    L.kin_peer_buffer_destroy.argtypes = [vp]
    L.kin_peer_grad_push.argtypes = [vp, i32, i32, i64, ctypes.POINTER(vp), i32, i32, u32, vp]
    L.kin_peer_grad_gather.argtypes = [vp, i32, i32, u32, vp, vp, vp, vp]
    for name in declared_functions():
        fn = getattr(L, name)  # raises AttributeError if the .so lacks a declared symbol
        if name not in ("kin_last_error_string", "kin_source_hash"):
            fn.restype = i32
    L.kin_source_hash.restype = ctypes.c_char_p
    if L.kin_abi_version() != define("KIN_ABI_VERSION"):
        raise KinError("libkin_b200.so ABI version does not match include/kin_b200.h; rebuild")
    _lib = L
    return L


def check(code: int) -> None:
    if code != 0:
        raise KinError(f"[{code}] {lib().kin_last_error_string().decode()}")
