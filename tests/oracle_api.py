"""ctypes binding of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE ONLY.

Nothing under daachorse_b200/ imports this module.  It is used by tests/, by
__graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "liboracle.so")

STANDARD, LEFTMOST_LONGEST, LEFTMOST_FIRST = 0, 1, 2
KIND = {"Standard": 0, "LeftmostLongest": 1, "LeftmostFirst": 2}
(FIND, FIND_OVERLAPPING, FIND_OVERLAPPING_NO_SUFFIX, LEFTMOST_FIND, FIND_STEPPER,
 FIND_OVERLAPPING_STEPPER) = range(6)
MODE = {
    "find_iter": FIND,
    "find_overlapping_iter": FIND_OVERLAPPING,
    "find_overlapping_no_suffix_iter": FIND_OVERLAPPING_NO_SUFFIX,
    "leftmost_find_iter": LEFTMOST_FIND,
    "find_stepper": FIND_STEPPER,
    "find_overlapping_stepper": FIND_OVERLAPPING_STEPPER,
}
OK, INVALID_ARGUMENT, AUTOMATON_SCALE, INVALID_CONVERSION, INVALID_AUTOMATON, MATCH_KIND_MISMATCH = range(6)

MATCH_DTYPE = np.dtype([("start", "<u4"), ("end", "<u4"), ("value", "<u4")])


class OracleError(Exception):
    def __init__(self, code):
        super().__init__("oracle status %d" % code)
        self.code = code


def build_oracle():
    """(Re)build liboracle.so from oracle/dach_oracle.c if it is missing or stale."""
    src = os.path.join(ORACLE_DIR, "dach_oracle.c")
    hdr = os.path.join(ORACLE_DIR, "dach_oracle.h")
    if (not os.path.exists(LIB_PATH)) or (
        os.path.exists(src) and os.path.getmtime(LIB_PATH) < max(os.path.getmtime(src), os.path.getmtime(hdr))
    ):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build_oracle()
    L = C.CDLL(LIB_PATH)
    vp, u8p, u32p, u64p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    L.orc_build.argtypes = [C.c_int, u8p, u64p, u32p, C.c_uint32, C.c_uint8, C.c_uint32, C.POINTER(vp)]
    L.orc_build.restype = C.c_int
    L.orc_free.argtypes = [vp]
    L.orc_free.restype = None
    L.orc_serialized_bytes.argtypes = [vp]
    L.orc_serialized_bytes.restype = C.c_size_t
    L.orc_serialize.argtypes = [vp, u8p, C.c_size_t]
    L.orc_serialize.restype = C.c_size_t
    L.orc_deserialize.argtypes = [C.c_int, u8p, C.c_size_t, C.POINTER(vp), C.POINTER(C.c_size_t)]
    L.orc_deserialize.restype = C.c_int
    for name, rt in [("orc_is_charwise", C.c_int), ("orc_match_kind", C.c_uint8),
                     ("orc_num_states", C.c_uint32), ("orc_heap_bytes", C.c_size_t),
                     ("orc_num_elements", C.c_size_t), ("orc_num_outputs", C.c_size_t),
                     ("orc_max_pattern_len", C.c_uint32), ("orc_alphabet_size", C.c_uint32)]:
        getattr(L, name).argtypes = [vp]
        getattr(L, name).restype = rt
    L.orc_peek_state.argtypes = [vp, C.c_size_t] + [C.POINTER(C.c_uint32)] * 4
    L.orc_peek_state.restype = C.c_int
    L.orc_mapper_get.argtypes = [vp, C.c_uint32]
    L.orc_mapper_get.restype = C.c_uint32
    L.orc_scan.argtypes = [vp, C.c_int, u8p, C.c_size_t, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.orc_scan.restype = C.c_int
    L.orc_utf8_next.argtypes = [u8p, C.POINTER(C.c_size_t)]
    L.orc_utf8_next.restype = C.c_uint32
    L.orc_scan_batch.argtypes = [vp, C.c_int, u8p, u64p, C.c_uint64, C.c_int, u64p, u64p, vp,
                                 C.c_uint64, C.POINTER(C.c_uint64)]
    L.orc_scan_batch.restype = C.c_int
    L.orc_hash_step.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
    L.orc_hash_step.restype = C.c_uint64
    _lib = L
    return L


def pack_patterns(patterns):
    """list of bytes/str -> (blob uint8 array, offsets uint64 array)."""
    bs = [p.encode("utf-8") if isinstance(p, str) else bytes(p) for p in patterns]
    offs = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        offs[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    blob = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if bs else np.zeros(0, dtype=np.uint8)
    return blob, offs


def _ptr(a):
    return a.ctypes.data if a is not None and a.size else None


class OraclePma:
    """One automaton held by the oracle."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def build(cls, patterns, charwise=False, match_kind=STANDARD, num_free_blocks=16, values=None):
        blob, offs = pack_patterns(patterns)
        return cls.build_packed(blob, offs, charwise, match_kind, num_free_blocks, values)

    @classmethod
    def build_packed(cls, blob, offs, charwise=False, match_kind=STANDARD, num_free_blocks=16, values=None):
        L = lib()
        h = C.c_void_p()
        vals = None if values is None else np.ascontiguousarray(values, dtype=np.uint32)
        n = len(offs) - 1
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        pad = blob if blob.size else np.zeros(1, dtype=np.uint8)
        rc = L.orc_build(int(bool(charwise)), pad.ctypes.data, offs.ctypes.data,
                         None if vals is None else (vals.ctypes.data if vals.size else None),
                         n, match_kind, num_free_blocks, C.byref(h))
        if rc != OK:
            raise OracleError(rc)
        return cls(h)

    @classmethod
    def deserialize(cls, data, charwise=False):
        L = lib()
        h = C.c_void_p()
        consumed = C.c_size_t()
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        pad = buf if buf.size else np.zeros(1, dtype=np.uint8)
        rc = L.orc_deserialize(int(bool(charwise)), pad.ctypes.data, buf.size, C.byref(h), C.byref(consumed))
        if rc != OK:
            raise OracleError(rc)
        return cls(h), consumed.value

    def __del__(self):
        try:
            if self._h:
                lib().orc_free(self._h)
                self._h = None
        except Exception:
            pass

    def serialize(self):
        L = lib()
        n = L.orc_serialized_bytes(self._h)
        buf = np.zeros(max(n, 1), dtype=np.uint8)
        L.orc_serialize(self._h, buf.ctypes.data, n)
        return buf[:n].tobytes()

    @property
    def charwise(self):
        return bool(lib().orc_is_charwise(self._h))

    def match_kind(self):
        return lib().orc_match_kind(self._h)

    def num_states(self):
        return lib().orc_num_states(self._h)

    def heap_bytes(self):
        return lib().orc_heap_bytes(self._h)

    def num_elements(self):
        return lib().orc_num_elements(self._h)

    def num_outputs(self):
        return lib().orc_num_outputs(self._h)

    def max_pattern_len(self):
        return lib().orc_max_pattern_len(self._h)

    def alphabet_size(self):
        return lib().orc_alphabet_size(self._h)

    def mapper_get(self, cp):
        r = lib().orc_mapper_get(self._h, cp)
        return None if r == 0xFFFFFFFF else r

    def peek(self, idx):
        vals = [C.c_uint32() for _ in range(4)]
        rc = lib().orc_peek_state(self._h, idx, *[C.byref(v) for v in vals])
        if rc:
            raise IndexError(idx)
        return tuple(v.value for v in vals)  # base, check, fail, output_pos

    def state_after(self, data, find_mode=False, state=0):
        """State id of the bytewise Standard automaton after consuming ``data`` from ``state`` with the
        transition function of src/bytewise.rs:1063-1088 (pure Python over peek(); small inputs only).
        ``find_mode``: FindStepper::consume, which returns to ROOT after a state with an output."""
        n = self.num_elements()
        cache = {}

        def st(i):
            if i not in cache:
                cache[i] = self.peek(i)
            return cache[i]

        for c in bytes(data):
            s = state
            while True:
                base = st(s)[0]
                if base != 0:
                    ci = base ^ c
                    if ci < n and st(ci)[1] == c:
                        s = ci
                        break
                if s == 0:
                    break
                s = st(s)[2]
            state = s
            if find_mode and st(state)[3] != 0:
                state = 0
        return state

    def scan(self, mode, haystack):
        """Returns a structured array of (start, end, value)."""
        L = lib()
        hay = haystack.encode("utf-8") if isinstance(haystack, str) else bytes(haystack)
        buf = np.frombuffer(hay, dtype=np.uint8)
        pad = buf if buf.size else np.zeros(1, dtype=np.uint8)
        n = C.c_size_t()
        cap = 64
        while True:
            out = np.zeros(cap, dtype=MATCH_DTYPE)
            rc = L.orc_scan(self._h, mode, pad.ctypes.data, buf.size, out.ctypes.data, cap, C.byref(n))
            if rc != OK:
                raise OracleError(rc)
            if n.value <= cap:
                return out[: n.value]
            cap = n.value

    def scan_triples(self, mode, haystack):
        """[(start, end, value), ...] as python ints."""
        r = self.scan(mode, haystack)
        return [(int(a), int(b), int(c)) for a, b, c in zip(r["start"], r["end"], r["value"])]

    def scan_batch(self, mode, text, offs, nthreads=1, want_matches=False, want_hashes=True):
        """Batch scan.  Returns dict(counts, hashes, total, matches)."""
        L = lib()
        text = np.ascontiguousarray(text, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        n = len(offs) - 1
        counts = np.zeros(max(n, 1), dtype=np.uint64)
        hashes = np.zeros(max(n, 1), dtype=np.uint64) if want_hashes else None
        total = C.c_uint64()
        pad = text if text.size else np.zeros(1, dtype=np.uint8)
        rc = L.orc_scan_batch(self._h, mode, pad.ctypes.data, offs.ctypes.data, n, nthreads,
                              counts.ctypes.data, None if hashes is None else hashes.ctypes.data,
                              None, 0, C.byref(total))
        if rc != OK:
            raise OracleError(rc)
        res = {"counts": counts[:n], "hashes": None if hashes is None else hashes[:n],
               "total": total.value, "matches": None}
        if want_matches:
            out = np.zeros(max(total.value, 1), dtype=MATCH_DTYPE)
            rc = L.orc_scan_batch(self._h, mode, pad.ctypes.data, offs.ctypes.data, n, nthreads,
                                  counts.ctypes.data, None, out.ctypes.data, total.value, C.byref(total))
            if rc != OK:
                raise OracleError(rc)
            res["matches"] = out[: total.value]
        return res


_native = None


def native_lib():
    """liboracle_native.so: the same source built with -march=native on this machine (the timed CPU baseline),
    in a temporary directory so that the tree is not written; falls back to the portable build if the machine
    has no compiler."""
    global _native
    if _native is None:
        try:
            with tempfile.TemporaryDirectory(prefix="dach_oracle_") as tmp:
                path = os.path.join(tmp, "liboracle_native.so")
                subprocess.check_call(["make", "-C", ORACLE_DIR, "-s", "native", "NATIVE_OUT=" + path],
                                      stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                L = C.CDLL(path)  # stays mapped after the directory is removed
        except Exception:
            L = lib()
        L.orc_bench_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p,
                                      C.POINTER(C.c_uint64)]
        L.orc_bench_batch.restype = C.c_int
        _native = L
    return _native


def bench_batch(pma, mode, text, offs, nthreads):
    """The timed CPU baseline (orc_bench_batch): returns the total match count."""
    L = native_lib()
    text = np.ascontiguousarray(text, dtype=np.uint8)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    total = C.c_uint64()
    rc = L.orc_bench_batch(pma._h, mode, text.ctypes.data, offs.ctypes.data, len(offs) - 1, int(nthreads), None, C.byref(total))
    if rc != OK:
        raise OracleError(rc)
    return int(total.value)


def hash_matches(matches, offs):
    """Per-haystack order-sensitive hashes of a result produced elsewhere (the GPU): structured or (k, 3)
    u32/i32 matches + n+1 offsets.  Comparable with scan_batch(...)["hashes"]."""
    m = np.ascontiguousarray(matches)
    if m.dtype != MATCH_DTYPE:
        m = np.ascontiguousarray(m.reshape(-1, 3)).view(np.uint32).reshape(-1).view(MATCH_DTYPE)
    offs = np.ascontiguousarray(offs, dtype=np.uint64)
    n = len(offs) - 1
    out = np.zeros(max(n, 1), dtype=np.uint64)
    L = lib()
    L.orc_hash_matches.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
    L.orc_hash_matches.restype = None
    pad = m if m.size else np.zeros(1, dtype=MATCH_DTYPE)
    L.orc_hash_matches(pad.ctypes.data, offs.ctypes.data, n, out.ctypes.data)
    return out[:n]


def cpu_budget():
    """How many CPUs this process may really use: the affinity mask, cut by the cgroup CPU quota if one is set
    (a container that sees 128 CPUs but is given 16 CPUs' worth of time runs 128 busy threads 8x slower)."""
    info = {"os_cpu_count": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["os_cpu_count"]
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    quota = q / per
            break
        except Exception:
            continue
    info["cgroup_cpu_quota"] = quota
    use = info["affinity"]
    if quota:
        use = max(1, min(use, int(quota + 0.5)))
    info["threads"] = use
    return info


def utf8_next(data, pos):
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    p = C.c_size_t(pos)
    cp = lib().orc_utf8_next(buf.ctypes.data, C.byref(p))
    return p.value, cp


def hash_tuples(triples):
    """Order-sensitive hash of [(start,end,value)...] (same fold as orc_hash_step)."""
    M = (1 << 64) - 1
    h = 0
    for s, e, v in triples:
        h ^= (s + 0x9E3779B97F4A7C15) & M
        h = (h * 0x100000001B3) & M
        h ^= (e + 0xC2B2AE3D27D4EB4F) & M
        h = (h * 0x100000001B3) & M
        h ^= (v + 0x165667B19E3779F9) & M
        h = (h * 0x100000001B3) & M
        h ^= h >> 29
    return h
