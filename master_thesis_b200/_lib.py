"""ctypes binding of libmt_b200.so (the C ABI declared in include/mt_b200.h).

The prototypes are parsed from the header, so the Python side can never drift
from the C declarations.  There is NO fallback: if the shared library is
missing or a call fails, a RuntimeError is raised (the product path must fail
loudly without its CUDA extension).
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HEADER = os.path.join(ROOT, "include", "mt_b200.h")
# MT_B200_LIB: developer knob for tuning sweeps (another build of the SAME library, see build.py)
LIB_PATH = os.environ.get("MT_B200_LIB") or os.path.join(HERE, "libmt_b200.so")

_CTYPES = {
    "int": ctypes.c_int,
    "int64_t": ctypes.c_int64,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
    "mt_stream_t": ctypes.c_void_p,
    "void *": ctypes.c_void_p,
    "const void *": ctypes.c_void_p,
    "float *": ctypes.c_void_p,
    "const float *": ctypes.c_void_p,
    "const uint8_t *": ctypes.c_void_p,
    "const int *": ctypes.c_void_p,
    "int *": ctypes.POINTER(ctypes.c_int),
    "const char *": ctypes.c_char_p,
}


def parse_header(path=HEADER):
    """Returns {name: (restype_str, [(argtype_str, argname), ...])} for every MT_API prototype."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = {}
    for m in re.finditer(r"MT_API\s+([\w\s\*]+?)\s*\b(mt_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3)
        ret = re.sub(r"\s+", " ", ret).replace(" *", " *")
        parsed = []
        args = args.strip()
        if args and args != "void":
            for a in args.split(","):
                a = re.sub(r"\s+", " ", a.strip())
                mm = re.match(r"(.*?)(\w+)$", a)
                parsed.append((mm.group(1).strip(), mm.group(2)))
        protos[name] = (ret, parsed)
    return protos


_lib = None
_protos = None


def load():
    """Loads the library (once) and attaches argtypes/restype to every entry point."""
    global _lib, _protos
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "master_thesis_b200: %s is missing - build it with "
            "`python -m master_thesis_b200.build` (nvcc, sm_100a). There is no CPU "
            "or PyTorch fallback for this path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    _protos = parse_header()
    for name, (ret, args) in _protos.items():
        fn = getattr(lib, name)          # AttributeError => header/library mismatch, loud
        fn.restype = _CTYPES[ret]
        fn.argtypes = [_CTYPES[t] for t, _ in args]
    _lib = lib
    return lib


def prototypes():
    load()
    return _protos


def last_error():
    return load().mt_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, last_error()))


_recording = None


def call(name, *args):
    """Calls an int-returning entry point and raises on a non-zero code.

    Inside ``record()`` the call is also appended, with its arguments already
    marshalled to ctypes, to the active ``Plan``."""
    fn = getattr(load(), name)
    rc = fn(*args)
    check(rc, name)
    if _recording is not None:
        cargs = tuple(a if (a is None or isinstance(a, ctypes._SimpleCData)) else t(a)
                      for t, a in zip(fn.argtypes, args))
        _recording.entries.append((name, fn, cargs))


class Plan(object):
    """A recorded sequence of C-ABI launches (same pointers, sizes and stream).

    Replaying costs one foreign call per entry and no tensor bookkeeping, so a
    launch-bound loop stays GPU-bound; ``Plan.__call__`` can also be captured into
    a CUDA graph.  The caller keeps the recorded inputs/outputs alive."""

    def __init__(self):
        self.entries = []
        self.keep = []      # every tensor allocated while recording: the plan owns its buffers

    def __call__(self):
        for name, fn, cargs in self.entries:
            rc = fn(*cargs)
            if rc:
                check(rc, name)

    def names(self):
        return [e[0] for e in self.entries]

    def args(self, i):
        """Arguments of entry ``i`` by the parameter names of the header (pointers as integers or None)."""
        name, _, cargs = self.entries[i]
        return {pname: (a.value if isinstance(a, ctypes._SimpleCData) else a)
                for (_, pname), a in zip(_protos[name][1], cargs)}

    def run_entry(self, i):
        name, fn, cargs = self.entries[i]
        rc = fn(*cargs)
        if rc:
            check(rc, name)


def keep(t):
    """Registers a tensor with the active recording (no-op otherwise) and returns it."""
    if _recording is not None and t is not None:
        _recording.keep.append(t)
    return t


class record(object):
    """``with record() as plan: step(...)`` - executes the step and records its launches."""

    def __enter__(self):
        global _recording
        if _recording is not None:
            raise RuntimeError("nested record()")
        _recording = Plan()
        return _recording

    def __exit__(self, *exc):
        global _recording
        _recording = None
        return False
