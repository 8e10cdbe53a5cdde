"""ctypes view of ``include/caengine.h``.

The struct layouts are parsed from the header at import time so that the header stays the single
source of truth for the ABI (a field added there is picked up here; a mismatch cannot happen
silently).  Only ``int32_t`` / ``int64_t`` / ``double`` scalars, arrays of them and ``const T*``
pointers appear in the ABI structs.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List, Tuple

REPO_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(REPO_ROOT, "include", "caengine.h")
PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ENGINE_LIB = os.path.join(PKG_DIR, "libcaengine.so")

_SCALARS = {"int32_t": C.c_int32, "int64_t": C.c_int64, "uint8_t": C.c_uint8,
            "uint32_t": C.c_uint32, "double": C.c_double, "size_t": C.c_size_t}


def _strip_comments(src: str) -> str:
    return re.sub(r"/\*.*?\*/", "", src, flags=re.S)


def _parse_struct(src: str, name: str) -> List[Tuple[str, object]]:
    m = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S)
    if not m:
        raise RuntimeError("struct %s not found in %s" % (name, HEADER))
    fields: List[Tuple[str, object]] = []
    for decl in m.group(1).split(";"):
        decl = decl.strip()
        if not decl:
            continue
        mm = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*([\w, ]+?)(\[(\d+)\])?$", decl)
        if not mm:
            raise RuntimeError("cannot parse field %r of %s" % (decl, name))
        ctype = _SCALARS[mm.group(2)]
        for fname in [f.strip() for f in mm.group(4).split(",")]:
            if mm.group(3):
                fields.append((fname, C.POINTER(ctype)))
            elif mm.group(6):
                fields.append((fname, ctype * int(mm.group(6))))
            else:
                fields.append((fname, ctype))
    return fields


def _parse_enums(src: str) -> Dict[str, int]:
    out: Dict[str, int] = {}
    for m in re.finditer(r"enum \w+ \{(.*?)\};", src, flags=re.S):
        nxt = 0
        for item in m.group(1).split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                k, v = [s.strip() for s in item.split("=")]
                nxt = int(v, 0)
            else:
                k = item
            out[k] = nxt
            nxt += 1
    for m in re.finditer(r"#define (CAE_\w+) (\d+)", src):
        out[m.group(1)] = int(m.group(2))
    return out


with open(HEADER) as _f:
    _SRC = _strip_comments(_f.read())

CONST = _parse_enums(_SRC)
globals().update(CONST)


class cae_objects(C.Structure):
    _fields_ = _parse_struct(_SRC, "cae_objects")


class cae_config(C.Structure):
    _fields_ = _parse_struct(_SRC, "cae_config")


class cae_stats(C.Structure):
    _fields_ = _parse_struct(_SRC, "cae_stats")


class cae_price_inputs(C.Structure):
    _fields_ = _parse_struct(_SRC, "cae_price_inputs")


def declared_functions() -> List[str]:
    """Names of every function the header declares (used by the symbol-export test)."""
    return sorted(set(re.findall(r"\b(cae_\w+)\s*\(", _SRC)))


REASON_NAMES = {v: k for k, v in CONST.items() if k.startswith("CAE_R_")}

# reason -> (plugin name, reason string) as the reference reports them
REASON_PLUGIN = {
    CONST["CAE_R_OK"]: ("", ""),
    CONST["CAE_R_PREFILTER_NODEAFFINITY"]: ("NodeAffinity", "PreFilter filtered the Node out"),
    CONST["CAE_R_NODE_UNSCHEDULABLE"]: ("NodeUnschedulable", "node(s) were unschedulable"),
    CONST["CAE_R_NODE_NAME"]: ("NodeName", "node(s) didn't match the requested node name"),
    CONST["CAE_R_TAINT"]: ("TaintToleration", "node(s) had untolerated taint(s)"),
    CONST["CAE_R_NODE_AFFINITY"]: ("NodeAffinity", "node(s) didn't match Pod's node affinity/selector"),
    CONST["CAE_R_NODE_PORTS"]: ("NodePorts", "node(s) didn't have free ports for the requested pod ports"),
    CONST["CAE_R_FIT"]: ("NodeResourcesFit", "Insufficient resources / Too many pods"),
    CONST["CAE_R_PTS_MISSING_LABEL"]: ("PodTopologySpread", "node(s) didn't match pod topology spread constraints (missing required label)"),
    CONST["CAE_R_PTS_SKEW"]: ("PodTopologySpread", "node(s) didn't match pod topology spread constraints"),
    CONST["CAE_R_IPA_AFFINITY"]: ("InterPodAffinity", "node(s) didn't match pod affinity rules"),
    CONST["CAE_R_IPA_ANTI_AFFINITY"]: ("InterPodAffinity", "node(s) didn't match pod anti-affinity rules"),
    CONST["CAE_R_IPA_EXISTING_ANTI_AFFINITY"]: ("InterPodAffinity", "node(s) didn't satisfy existing pods anti-affinity rules"),
}

_engine_lib = None


def load_engine_lib() -> C.CDLL:
    """dlopen the product library.  Fails loudly: there is NO CPU fallback in the product path."""
    global _engine_lib
    if _engine_lib is not None:
        return _engine_lib
    path = os.environ.get("CAE_ENGINE_LIB", ENGINE_LIB)     # experiments: another build of the same library
    if not os.path.exists(path):
        raise RuntimeError(
            "libcaengine.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'`. The engine has no CPU fallback." % path)
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    P = C.POINTER
    lib.cae_create.argtypes = [P(cae_config), P(C.c_void_p)]
    lib.cae_create.restype = C.c_int32
    lib.cae_destroy.argtypes = [C.c_void_p]
    lib.cae_destroy.restype = None
    lib.cae_last_error.restype = C.c_char_p
    lib.cae_version.restype = C.c_char_p
    lib.cae_load.argtypes = [C.c_void_p, P(cae_objects)]
    lib.cae_load.restype = C.c_int32
    lib.cae_load_pending.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
    lib.cae_load_pending.restype = C.c_int32
    lib.cae_feasibility.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cae_feasibility.restype = C.c_int32
    lib.cae_feasibility_groups.argtypes = [C.c_void_p, C.c_void_p]
    lib.cae_feasibility_groups.restype = C.c_int32
    lib.cae_estimate_all.argtypes = [C.c_void_p] + [C.c_void_p] * 5
    lib.cae_estimate_all.restype = C.c_int32
    lib.cae_estimate_all_ex.argtypes = [C.c_void_p] + [C.c_void_p] * 7
    lib.cae_estimate_all_ex.restype = C.c_int32
    lib.cae_expander_best.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cae_expander_best.restype = C.c_int32
    lib.cae_get_stats.argtypes = [C.c_void_p, P(cae_stats)]
    lib.cae_get_stats.restype = C.c_int32
    lib.cae_peer_handle.argtypes = [C.c_void_p, C.c_void_p]
    lib.cae_peer_handle.restype = C.c_int32
    lib.cae_peer_attach.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
    lib.cae_peer_attach.restype = C.c_int32
    lib.cae_device_buffer.argtypes = [C.c_void_p, C.c_int32, P(C.c_size_t)]
    lib.cae_device_buffer.restype = C.c_void_p
    lib.cae_filter_schedulable.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                           C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cae_filter_schedulable.restype = C.c_int32
    lib.cae_simulate_removals.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p] * 5 + [C.c_int32] * 3 + [C.c_void_p, C.c_int32] + \
        [C.c_void_p] * 4
    lib.cae_simulate_removals.restype = C.c_int32
    lib.cae_price_scores.argtypes = [C.c_void_p, P(cae_price_inputs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cae_price_scores.restype = C.c_int32
    lib.cae_expander_chain_ex.argtypes = [C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 7
    lib.cae_expander_chain_ex.restype = C.c_int32
    lib.cae_waste_scores.argtypes = [C.c_void_p, C.c_void_p]
    lib.cae_waste_scores.restype = C.c_int32
    lib.cae_expander_chain.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cae_expander_chain.restype = C.c_int32
    lib.cae_stream.argtypes = [C.c_void_p]
    lib.cae_stream.restype = C.c_void_p
    _engine_lib = lib
    return lib
