"""ctypes binding of libusv_b200.so (the C ABI declared in include/usv_b200.h).

The ctypes Structures are generated from the header itself at import time, so the Python mirror
cannot drift from the C layout; the library additionally reports sizeof() for each struct and the
loader refuses to run on a mismatch.  There is no CPU fallback: if the shared library is missing
this module raises, and every compute call needs CUDA tensors.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(_ROOT, "include", "usv_b200.h")
LIB_PATH = os.environ.get("USV_B200_LIB", os.path.join(_HERE, "lib", "libusv_b200.so"))

_CTYPES = {
    "float": ctypes.c_float, "int32_t": ctypes.c_int32, "uint32_t": ctypes.c_uint32,
    "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64,
    "float*": ctypes.c_void_p, "const float*": ctypes.c_void_p, "int64_t*": ctypes.c_void_p,
    "uint32_t*": ctypes.c_void_p, "int32_t*": ctypes.c_void_p, "double*": ctypes.c_void_p,
    "uint64_t*": ctypes.c_void_p, "const int32_t*": ctypes.c_void_p, "const uint64_t*": ctypes.c_void_p,
    "const uint8_t*": ctypes.c_void_p, "uint8_t*": ctypes.c_void_p,
}


def _strip_comments(src: str) -> str:
    return re.sub(r"/\*.*?\*/", "", src, flags=re.S)


def _parse_structs(src: str) -> Dict[str, type]:
    """Turns every `typedef struct { ... } Name;` of the header into a ctypes.Structure."""
    src = _strip_comments(src)
    out: Dict[str, type] = {}
    for m in re.finditer(r"typedef\s+struct\s*\{(.*?)\}\s*(\w+)\s*;", src, flags=re.S):
        body, name = m.group(1), m.group(2)
        fields = []
        for decl in body.split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            mm = re.match(r"((?:const\s+)?\w+\s*\*?)\s*(.*)", decl)
            ctype_name, rest = mm.group(1).replace(" *", "*").strip(), mm.group(2)
            if ctype_name.endswith("*") or rest.startswith("*"):
                base = ctype_name.rstrip("*").strip() + "*"
                ctype = _CTYPES[base]
                rest = rest.lstrip("* ")
            elif ctype_name in out:
                ctype = out[ctype_name]
            else:
                ctype = _CTYPES[ctype_name]
            for var in rest.split(","):
                var = var.strip().lstrip("*").strip()
                am = re.match(r"(\w+)\[(\d+)\]", var)
                if am:
                    fields.append((am.group(1), ctype * int(am.group(2))))
                else:
                    fields.append((var, ctype))
        out[name] = type(name, (ctypes.Structure,), {"_fields_": fields})
    return out


def _parse_enums(src: str) -> Dict[str, int]:
    src = _strip_comments(src)
    vals: Dict[str, int] = {}
    for m in re.finditer(r"#define\s+((?:USV|PPO)_\w+)\s+(\d+)", src):
        vals[m.group(1)] = int(m.group(2))
    for m in re.finditer(r"enum\s*\{(.*?)\}\s*;", src, flags=re.S):
        cur = -1
        for item in m.group(1).split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                k, v = [x.strip() for x in item.split("=")]
                # integer literal or an arithmetic expression over earlier constants of this header
                cur = int(eval(v, {"__builtins__": {}}, dict(vals)))
            else:
                k, cur = item, cur + 1
            vals[k] = cur
    return vals


with open(HEADER) as _f:
    _SRC = _f.read()
STRUCTS = _parse_structs(_SRC)
ENUMS = _parse_enums(_SRC)
UsvHydrostaticsParams = STRUCTS["UsvHydrostaticsParams"]
UsvHydrodynamicsParams = STRUCTS["UsvHydrodynamicsParams"]
UsvPenaltyTerm = STRUCTS["UsvPenaltyTerm"]
UsvStepParams = STRUCTS["UsvStepParams"]
UsvEnvBuffers = STRUCTS["UsvEnvBuffers"]
UsvLiveParams = STRUCTS["UsvLiveParams"]
UsvLiveBuffers = STRUCTS["UsvLiveBuffers"]
PpoLossParams = STRUCTS["PpoLossParams"]
PpoAdamParams = STRUCTS["PpoAdamParams"]
PpoPeerComm = STRUCTS["PpoPeerComm"]
UsvCaptureXYIO = STRUCTS["UsvCaptureXYIO"]

_lib = None


class UsvLibraryError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Loads libusv_b200.so (built by __graft_entry__.build() / csrc/Makefile).  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UsvLibraryError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU / torch fallback for the USV hot path)")
    L = ctypes.CDLL(LIB_PATH)
    L.usv_b200_error_string.restype = ctypes.c_char_p
    L.usv_b200_launch_count.restype = ctypes.c_int64
    L.usv_b200_sizeof.restype = ctypes.c_int64
    L.usv_b200_sizeof.argtypes = [ctypes.c_char_p]
    L.ppo_param_count.restype = ctypes.c_int64
    L.ppo_train_scratch_floats.restype = ctypes.c_int64
    L.ppo_train_tc_workspace_floats.restype = ctypes.c_int64
    L.ppo_packed_weight_floats.restype = ctypes.c_int64
    L.usv_live_scene_workspace_bytes.restype = ctypes.c_int64
    L.ppo_peer_window_bytes.restype = ctypes.c_int64
    L.ppo_minibatch_step_peer_entries.restype = ctypes.c_int64
    L.ppo_loopz_peer_entries.restype = ctypes.c_int64
    L.dagger_history_encoder_param_count.restype = ctypes.c_int64
    L.dagger_train_scratch_floats.restype = ctypes.c_int64
    L.usv_live_scene_workspace_bytes.argtypes = [ctypes.c_int64]
    for name, st in STRUCTS.items():
        want = L.usv_b200_sizeof(name.encode())
        if want != ctypes.sizeof(st):
            raise UsvLibraryError(f"ABI mismatch for {name}: header says {ctypes.sizeof(st)} B, library {want} B")
    if L.usv_b200_abi_version() != ENUMS["USV_B200_ABI_VERSION"]:
        raise UsvLibraryError("ABI version mismatch between include/usv_b200.h and libusv_b200.so")
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().usv_b200_error_string(ctypes.c_int(rc)).decode()
        raise RuntimeError(f"libusv_b200 {what} failed: [{rc}] {msg}")


def launch_count() -> int:
    return int(lib().usv_b200_launch_count())


def ptr(t: torch.Tensor | None, dtype=None) -> ctypes.c_void_p:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return ctypes.c_void_p(0)
    if not t.is_cuda:
        raise UsvLibraryError("libusv_b200 needs CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise ValueError("libusv_b200 needs contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if t.device.index != torch._C._cuda_getDevice():
        # stream() hands the kernels the CURRENT device's stream: a tensor of another device would be launched on the wrong GPU
        raise UsvLibraryError(f"tensor lives on {t.device} but the current CUDA device is {torch._C._cuda_getDevice()}: wrap the call in "
                              "torch.cuda.device(...) or call torch.cuda.set_device() first (one process per GPU)")
    return ctypes.c_void_p(t.data_ptr())


def stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def exported_symbols():
    """Every function the header declares (used by the CPU test that the library exports them all)."""
    src = _strip_comments(_SRC)
    return sorted(set(re.findall(r"\b((?:usv|ppo)_\w+)\s*\(", src)))
