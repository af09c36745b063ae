"""ctypes binding of libmdvit_b200.so (the C ABI declared in include/mdvit_b200.h).

There is no fallback: if the shared library is missing or a call fails, this raises."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MDV_LIB_PATH") or os.path.join(_HERE, "libmdvit_b200.so")   # (override: A/B builds during development)

c_void_p, c_int, c_float, c_uint32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_uint32

ACT_NONE, ACT_GELU, ACT_RELU, ACT_HSWISH = 0, 1, 2, 3


class GemmEpi(ctypes.Structure):
    _fields_ = [
        ("bias", c_void_p), ("residual", c_void_p), ("mul_gelu_grad", c_void_p), ("out_preact", c_void_p),
        ("out", c_void_p), ("rowscale", c_void_p), ("rng", c_void_p), ("colsum", c_void_p), ("colscale", c_void_p),
        ("ld_res", c_int), ("ld_mul", c_int), ("ld_preact", c_int), ("ldc", c_int),
        ("rows_per_scale", c_int), ("out_bf16", c_int), ("act", c_int), ("accumulate", c_int), ("preact_mode", c_int), ("mul_mode", c_int),
        ("dropout_p", c_float), ("drop_stream", c_uint32),
    ]


MAX_GROUPS = 8      # MDV_MAX_GROUPS


class PtrTable(ctypes.Structure):
    """MdvPtrTable: one device pointer per row group (G <= MAX_GROUPS), passed by value."""
    _fields_ = [("p", c_void_p * MAX_GROUPS)]


def ptr_table(tensors):
    """PtrTable of the tensors' device pointers (None entries -> NULL)."""
    if len(tensors) > MAX_GROUPS:
        raise ValueError(f"at most {MAX_GROUPS} groups")
    t = PtrTable()
    for i, x in enumerate(tensors):
        t.p[i] = None if x is None else x.data_ptr()
    return t


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(mdvit_b200 has no CPU or PyTorch fallback path)")
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in header_signatures().items():
            fn = getattr(_lib, name)          # AttributeError here == header/library mismatch
            fn.restype, fn.argtypes = restype, argtypes
        if _PROFILE:
            _lib = _ProfiledLib(_lib)
    return _lib


_PROFILE = bool(int(os.environ.get("MDV_PROFILE", "0")))
PROFILE_LOG = []     # (key, start_event, end_event) per C-ABI call when MDV_PROFILE=1 (development aid only)


class _ProfiledLib:
    """Wraps every mdv_* entry point with CUDA events on the launching stream; keys calls by their integer arguments."""

    def __init__(self, raw):
        self._raw = raw

    def __getattr__(self, name):
        fn = getattr(self._raw, name)
        if not name.startswith("mdv_") or name in ("mdv_launch_count", "mdv_version", "mdv_attn_stats_floats", "mdv_gemm_tune"):
            return fn

        def wrapped(*args):
            key = [name]
            for a in args:
                if isinstance(a, bool) or isinstance(a, int):
                    key.append(int(a))
                elif isinstance(a, float):
                    key.append(round(a, 4))
                elif hasattr(a, "_obj") and isinstance(a._obj, GemmEpi):
                    e = a._obj
                    key.append("epi[" + ",".join(k for k, v in (("bias", e.bias), ("res", e.residual), ("mulg", e.mul_gelu_grad),
                                                                ("pre", e.out_preact), ("rs", e.rowscale), ("drop", e.dropout_p > 0),
                                                                ("bf16" if e.out_bf16 else "f32", True), ("act%d" % e.act, e.act)) if v) + "]")
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            rc = fn(*args)
            t.record()
            PROFILE_LOG.append((tuple(key), s, t))
            return rc

        setattr(self, name, wrapped)
        return wrapped


def profile_report(top=80, clear=True):
    """Aggregate PROFILE_LOG by (entry point, integer args): total ms, calls, average us."""
    torch.cuda.synchronize()
    agg = {}
    for key, s, t in PROFILE_LOG:
        a = agg.setdefault(key, [0, 0.0])
        a[0] += 1
        a[1] += s.elapsed_time(t)
    if clear:
        PROFILE_LOG.clear()
    tot = sum(v[1] for v in agg.values())
    lines = [f"total {tot:.2f} ms over {sum(v[0] for v in agg.values())} calls"]
    for key, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:top]:
        lines.append(f"{ms:9.3f} ms {100 * ms / tot:5.1f}%  n={n:4d}  avg {ms / n * 1e3:8.1f} us  {key[0]} {' '.join(map(str, key[1:]))}")
    return "\n".join(lines)


HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "mdvit_b200.h")
_CTYPES = {"int": c_int, "float": c_float, "double": ctypes.c_double, "long long": ctypes.c_longlong,
           "uint32_t": c_uint32, "void": None, "MdvPtrTable": PtrTable}


def header_signatures(path=HEADER_PATH):
    """Parse include/mdvit_b200.h -> {name: (restype, [argtypes])}; every pointer is passed as void*."""
    import re
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    sigs = {}
    for m in re.finditer(r"\b(int|long long)\s+(mdv_\w+)\s*\(([^;{}]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), " ".join(m.group(3).split())
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(c_void_p)
                else:
                    base = a.replace("const ", "").rsplit(" ", 1)[0].strip()
                    argtypes.append(_CTYPES[base])
        sigs[name] = (_CTYPES[ret], argtypes)
    return sigs


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


class MdvError(RuntimeError):
    pass


_DEBUG_SYNC = bool(int(os.environ.get("MDV_DEBUG_SYNC", "0")))


def check(rc, what):
    if _DEBUG_SYNC and rc == 0:
        try:
            torch.cuda.synchronize()
        except Exception as ex:  # pragma: no cover - debug aid
            raise MdvError(f"{what}: asynchronous CUDA failure: {ex}") from ex
    if rc != 0:
        if rc > 0:
            msg = f"CUDA error {rc}"
        else:
            msg = {-1: "invalid argument", -2: "unsupported shape", -3: "driver entry point unavailable"}.get(rc, str(rc))
        raise MdvError(f"{what} failed: {msg}")
