"""ctypes binding of libpn12_b200.so (the C ABI declared in include/pn12_b200.h).

There is no CPU fallback and no alternative backend: if the library is missing or a call fails,
a RuntimeError is raised.  Pointers come from `tensor.data_ptr()`, the stream from
`torch.cuda.current_stream()`, so every call is asynchronous and CUDA-graph capturable.
"""
from __future__ import annotations

import ctypes as C
import os
import re

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libpn12_b200.so")
HEADER = os.path.join(os.path.dirname(PKG), "include", "pn12_b200.h")

_lib = None

# The C spellings include/pn12_b200.h may use.  Every pointer is passed as c_void_p: the header's types cannot tell host
# from device pointers, and c_void_p takes an integer address (data_ptr()) as well as a byref() or a ctypes array.
_SCALARS = {"int": C.c_int, "int32_t": C.c_int, "int64_t": C.c_int64, "size_t": C.c_size_t, "float": C.c_float}
_RETURNS = {"int": C.c_int, "size_t": C.c_size_t, "const char*": C.c_char_p}


def _spelling(t: str) -> str:
    return re.sub(r"\s*\*", "*", " ".join(t.split()))


def parse_header(text: str):
    """(integer #defines, structs: name -> ctypes.Structure, functions: name -> (argtypes, restype)) of a header written
    in the small C grammar of include/pn12_b200.h.  Anything outside it raises a ValueError naming the declaration."""
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"#ifdef __cplusplus.*?#endif", "", text, flags=re.S)
    consts = {k: int(v) for k, v in re.findall(r"^\s*#\s*define\s+(\w+)\s+(-?\d+)\s*$", text, flags=re.M)}
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    decl_re = r"[^;{}]*(?:\{[^{}]*\}[^;{}]*)?;"
    rest = re.sub(decl_re, "", text).strip()
    if rest:
        raise ValueError(f"cannot parse declaration: {rest}")
    types, structs, functions = dict(_SCALARS), {}, {}

    def var(s: str, decl: str):  # "T name" or "T name[N]" -> (name, ctype, spelling of T)
        m = re.fullmatch(r"(.*?)\s*\b(\w+)\s*(?:\[\s*(\w+)\s*\])?", s.strip())
        spelling = _spelling(m.group(1)) if m else ""
        t = C.c_void_p if "*" in spelling else types.get(spelling)
        if t is None:
            raise ValueError(f"unsupported type in {s.strip()!r} of: {decl}")
        if m.group(3):
            n = int(m.group(3)) if m.group(3).isdigit() else consts.get(m.group(3))
            if n is None:
                raise ValueError(f"unknown array bound {m.group(3)!r} in: {decl}")
            t = t * n
        return m.group(2), t, spelling

    for decl in (" ".join(d[:-1].split()) for d in re.findall(decl_re, text)):
        if not decl or re.fullmatch(r"enum \w+ \{[^{}]*\}", decl):
            continue
        if m := re.fullmatch(r"typedef struct (\w+) \{([^{}]*)\} \1", decl):
            fields = []
            for field in (f for f in m.group(2).split(";") if f.strip()):
                first, *more = field.split(",")
                name, t, spelling = var(first, decl)
                if more and "*" in spelling:
                    raise ValueError(f"one pointer field per declaration in: {decl}")
                fields += [(name, t)] + [var(f"{spelling} {v}", decl)[:2] for v in more]
            structs[m.group(1)] = type(m.group(1), (C.Structure,), {"_fields_": fields})
        elif m := re.fullmatch(r"typedef ([^{}\[\]]+)", decl):
            name, t, _ = var(m.group(1), decl)
            types[name] = t
        elif m := re.fullmatch(r"(.+?) ?\b(pn_\w+) ?\(([^\[\]]*)\)", decl):
            restype = _RETURNS.get(_spelling(m.group(1)))
            if restype is None:
                raise ValueError(f"unsupported return type in: {decl}")
            params = [] if m.group(3).strip() == "void" else m.group(3).split(",")
            functions[m.group(2)] = ([var(p, decl)[1] for p in params], restype)
        else:
            raise ValueError(f"cannot parse declaration: {decl}")
    return consts, structs, functions


with open(HEADER) as _f:
    _CONSTS, _STRUCTS, _FUNCTIONS = parse_header(_f.read())
MLP_MAX_LAYERS = _CONSTS["PN_MLP_MAX_LAYERS"]
LaunchOpts = _STRUCTS["pn_launch_opts"]           # per-call launch options (all zeros = defaults)
MlpDesc = _STRUCTS["pn_mlp_desc"]
TrainPackItem = _STRUCTS["pn_train_pack_item"]


def declared_symbols() -> list:
    """Every function name include/pn12_b200.h declares (used by the export test)."""
    return sorted(_FUNCTIONS)


def lib():
    """Load the library once; fail loudly when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m pointnet12_b200.build` "
                "(nvcc, sm_100a). pointnet12_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in _FUNCTIONS.items():
            fn = getattr(handle, name)
            fn.argtypes, fn.restype = argtypes, restype
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().pn_last_error_string().decode("utf-8", "replace")
        kind = "CUDA error" if status > 0 else "argument error"
        raise RuntimeError(f"{what} failed ({kind} {status}): {msg}")


# ---- launch accounting (used by bench.py): how many of our kernels were launched, and optional CUDA-event
# timing of selected entry points on the launching stream.
launch_count = 0
_timed = {}          # name -> list of (start_event, stop_event, tag)


def time_entry_points(names=None):
    """Enable (names = iterable of entry points) or disable (None) CUDA-event timing; returns the old records."""
    global _timed
    old, _timed = _timed, ({n: [] for n in names} if names else {})
    return old


def call(name: str, *args, tag=None) -> None:
    global launch_count
    launch_count += 1
    rec = _timed.get(name)
    if rec is None:
        check(getattr(lib(), name)(*args), name)
        return
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    check(getattr(lib(), name)(*args), name)
    b.record()
    rec.append((a, b, tag))
