"""ctypes binding of the C ABI in include/holo_spf.h (libholo_spf.so).

This is the Python twin of the `extern "C"` block a holo maintainer would add
(INTEGRATION.md).  It only marshals numpy arrays across the boundary; every
result is produced by the CUDA kernels behind the ABI.  If the shared library is
missing the import fails loudly — there is no Python/CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from contextlib import contextmanager
from dataclasses import dataclass
from pathlib import Path

import numpy as np

from .build import PRODUCT_LIB

HSPF_OK = 0
HSPF_E_INVAL = -1
HSPF_E_CUDA = -2
HSPF_E_NOMEM = -3
HSPF_E_NEEDS_ORACLE = -4
HSPF_E_UNSUPPORTED = -5
HSPF_E_JOB_STATUS = -6

VF_HOP = 0x01
VF_LEAF = 0x02
VF_LEAF_UNLESS_ROOT = 0x04
GF_NOHOP_TARGET_NO_NEXTHOP = 0x01
GF_HOPCOUNT = 0x02
COST_DISABLED = 0xFFFFFFFF
DIST_INF = 0xFFFFFFFF
NO_PARENT = 0xFFFFFFFF
JS_SATURATED = 0x1
JS_TOO_MANY_ATOMS = 0x2
JS_ORDER = 0x4
JS_INVALID = 0x8
JS_INTERNAL = 0x10
JS_NARROW = 0x20
RUN_DEVICE_PTRS = 0x1
MAX_OVERRIDES = 8
PATHS = {"auto": 0, "general": 1, "general_kahn": 2}   # hspf_debug_set_path

_u32p = C.POINTER(C.c_uint32)
_u16p = C.POINTER(C.c_uint16)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)


class CsrStruct(C.Structure):
    _fields_ = [
        ("n_vertices", C.c_uint32),
        ("n_edges", C.c_uint32),
        ("row_ptr", _u32p),
        ("col", _u32p),
        ("cost", _u32p),
        ("vflags", _u8p),
        ("reject_above", C.c_uint32),
        ("saturate_at", C.c_uint32),
        ("flags", C.c_uint32),
        ("delta", C.c_uint32),
    ]


class JobsStruct(C.Structure):
    _fields_ = [
        ("n_jobs", C.c_uint32),
        ("roots", _u32p),
        ("ov_off", _u32p),
        ("ov_edge", _u32p),
        ("ov_cost", _u32p),
    ]


class ResultStruct(C.Structure):
    _fields_ = [
        ("dist", _u32p),
        ("hops", _u16p),
        ("first_parent", _u32p),
        ("n_parents", _u16p),
        ("nh_mask", _u64p),
        ("nh_words", C.c_uint32),
        ("job_status", _u32p),
    ]


class Result16Struct(C.Structure):
    _fields_ = [
        ("dist", _u16p),
        ("hops", _u16p),
        ("first_parent", _u16p),
        ("n_parents", _u16p),
        ("nh_mask", _u16p),
        ("job_status", _u32p),
    ]


EXPORTS = [
    "hspf_version", "hspf_ctx_create", "hspf_ctx_destroy", "hspf_last_error",
    "hspf_graph_upload", "hspf_graph_free", "hspf_run_batch", "hspf_run_batch_async",
    "hspf_sync", "hspf_stream", "hspf_launch_count", "hspf_atom_decode", "hspf_atom_count",
    "hspf_ctx_reserve_sms", "hspf_debug_quad_image", "hspf_debug_phase_profile",
    "hspf_run_batch16", "hspf_run_batch16_async", "hspf_graph_info",
    "hspf_xchg_create", "hspf_xchg_attach", "hspf_xchg_slot", "hspf_xchg_slot_bytes", "hspf_xchg_acquire",
    "hspf_xchg_push", "hspf_xchg_wait", "hspf_xchg_release", "hspf_xchg_consumer_stream", "hspf_xchg_sync",
    "hspf_xchg_last_error", "hspf_xchg_destroy", "hspf_xchg_attach_ptr", "hspf_xchg_base", "hspf_xchg_set_push_bytes",
    "hspf_xchg_acquire_direct", "hspf_xchg_peer_deltas", "hspf_xchg_publish", "hspf_ctx_set_peer_slots",
    "hspf_graph_update_costs", "hspf_debug_set_path",
]


class HspfError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"hspf error {code}: {msg}")
        self.code = code


_lib = None


def load_library(path: Path | None = None) -> C.CDLL:
    """Load libholo_spf.so (built in-tree by holo_b200.build); fail loudly."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else PRODUCT_LIB
    if not p.exists():
        raise ImportError(
            f"{p} is missing: build it with `python -m holo_b200.build` "
            "(there is no CPU fallback for the SPF engine)")
    lib = C.CDLL(str(p))
    lib.hspf_version.restype = C.c_char_p
    lib.hspf_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.hspf_ctx_destroy.argtypes = [C.c_void_p]
    lib.hspf_ctx_destroy.restype = None
    lib.hspf_last_error.argtypes = [C.c_void_p]
    lib.hspf_last_error.restype = C.c_char_p
    lib.hspf_graph_upload.argtypes = [C.c_void_p, C.POINTER(CsrStruct), C.POINTER(C.c_void_p)]
    lib.hspf_graph_free.argtypes = [C.c_void_p, C.c_void_p]
    lib.hspf_graph_free.restype = None
    lib.hspf_run_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(JobsStruct), C.POINTER(ResultStruct), C.c_uint32]
    lib.hspf_run_batch_async.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(JobsStruct), C.POINTER(ResultStruct)]
    lib.hspf_sync.argtypes = [C.c_void_p]
    lib.hspf_stream.argtypes = [C.c_void_p]
    lib.hspf_stream.restype = C.c_void_p
    lib.hspf_launch_count.argtypes = [C.c_void_p]
    lib.hspf_launch_count.restype = C.c_uint64
    lib.hspf_ctx_reserve_sms.argtypes = [C.c_void_p, C.c_int]
    lib.hspf_atom_decode.argtypes = [C.POINTER(CsrStruct), C.c_uint32, C.c_uint32, _u32p, _u32p]
    lib.hspf_atom_count.argtypes = [C.POINTER(CsrStruct), C.c_uint32, _u32p]
    lib.hspf_debug_quad_image.argtypes = [C.POINTER(CsrStruct), C.POINTER(C.c_uint32), _u32p, _u32p, _u16p, _u16p,
                                          _u32p, _u32p, _u32p, _u32p]
    lib.hspf_debug_phase_profile.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_uint64)]
    lib.hspf_debug_set_path.argtypes = [C.c_void_p, C.c_int]
    lib.hspf_run_batch16.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(JobsStruct), C.POINTER(Result16Struct), C.c_uint32]
    lib.hspf_run_batch16_async.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(JobsStruct), C.POINTER(Result16Struct)]
    lib.hspf_graph_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint32)]
    if path is None:
        _lib = lib
    return lib


def _ptr(a: np.ndarray | None, ty):
    if a is None:
        return C.cast(None, ty)
    return a.ctypes.data_as(ty)


@dataclass
class Csr:
    """Host-side flattened graph (see hspf_csr in include/holo_spf.h)."""
    row_ptr: np.ndarray
    col: np.ndarray
    cost: np.ndarray
    vflags: np.ndarray
    reject_above: int = 0xFFFFFFFE
    saturate_at: int = 0
    flags: int = 0
    delta: int = 0

    def __post_init__(self):
        self.row_ptr = np.ascontiguousarray(self.row_ptr, dtype=np.uint32)
        self.col = np.ascontiguousarray(self.col, dtype=np.uint32)
        self.cost = np.ascontiguousarray(self.cost, dtype=np.uint32)
        self.vflags = np.ascontiguousarray(self.vflags, dtype=np.uint8)

    @property
    def n_vertices(self) -> int:
        return len(self.row_ptr) - 1

    @property
    def n_edges(self) -> int:
        return len(self.col)

    def as_struct(self) -> CsrStruct:
        s = CsrStruct()
        s.n_vertices = self.n_vertices
        s.n_edges = self.n_edges
        s.row_ptr = _ptr(self.row_ptr, _u32p)
        s.col = _ptr(self.col, _u32p)
        s.cost = _ptr(self.cost, _u32p)
        s.vflags = _ptr(self.vflags, _u8p)
        s.reject_above = self.reject_above
        s.saturate_at = self.saturate_at
        s.flags = self.flags
        s.delta = self.delta
        return s


@dataclass
class SpfResult:
    dist: np.ndarray          # [n_jobs, V] uint32
    hops: np.ndarray          # [n_jobs, V] uint16
    first_parent: np.ndarray  # [n_jobs, V] uint32
    n_parents: np.ndarray     # [n_jobs, V] uint16
    nh_mask: np.ndarray       # [n_jobs, V, nh_words] uint64
    job_status: np.ndarray    # [n_jobs] uint32
    status: int = 0           # return code of hspf_run_batch (0 or HSPF_E_JOB_STATUS)


def make_jobs(roots, overrides=None):
    """roots: sequence of vertex ids; overrides: optional list (per job) of
    [(edge, cost), ...].  Returns (JobsStruct, keepalive)."""
    roots = np.ascontiguousarray(roots, dtype=np.uint32)
    js = JobsStruct()
    js.n_jobs = len(roots)
    js.roots = _ptr(roots, _u32p)
    keep = [roots]
    if overrides is not None:
        off = np.zeros(len(roots) + 1, dtype=np.uint32)
        ed, co = [], []
        for j, ov in enumerate(overrides):
            for e, c in ov:
                ed.append(e)
                co.append(c)
            off[j + 1] = len(ed)
        ed = np.asarray(ed if ed else [0], dtype=np.uint32)
        co = np.asarray(co if co else [0], dtype=np.uint32)
        js.ov_off = _ptr(off, _u32p)
        js.ov_edge = _ptr(ed, _u32p)
        js.ov_cost = _ptr(co, _u32p)
        keep += [off, ed, co]
    return js, keep


class Graph:
    def __init__(self, ctx: "Context", handle: C.c_void_p, csr: Csr):
        self.ctx = ctx
        self.handle = handle
        self.csr = csr

    def free(self):
        if self.handle:
            self.ctx.lib.hspf_graph_free(self.ctx.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One engine context (one per protocol instance in the reference's threading
    model, holo-protocol/src/lib.rs:405-408)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.hspf_ctx_create(device, C.byref(h))
        if rc != HSPF_OK:
            raise HspfError(rc, "hspf_ctx_create failed (no usable CUDA device?)")
        self.handle = h
        self.device = device

    def close(self):
        if self.handle:
            self.lib.hspf_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def last_error(self) -> str:
        return self.lib.hspf_last_error(self.handle).decode()

    def _check(self, rc: int, allow=()):
        if rc != HSPF_OK and rc not in allow:
            raise HspfError(rc, self.last_error())
        return rc

    def upload(self, csr: Csr) -> Graph:
        s = csr.as_struct()
        h = C.c_void_p()
        self._check(self.lib.hspf_graph_upload(self.handle, C.byref(s), C.byref(h)))
        return Graph(self, h, csr)

    def run(self, graph: Graph, roots, overrides=None, nh_words: int = 1) -> SpfResult:
        """Host-pointer call: H2D of the job list, kernel, D2H of every plane."""
        js, keep = make_jobs(roots, overrides)
        n, V = js.n_jobs, graph.csr.n_vertices
        res = SpfResult(
            dist=np.empty((n, V), np.uint32), hops=np.empty((n, V), np.uint16),
            first_parent=np.empty((n, V), np.uint32), n_parents=np.empty((n, V), np.uint16),
            nh_mask=np.empty((n, V, nh_words), np.uint64), job_status=np.zeros(n, np.uint32))
        rs = ResultStruct()
        rs.dist = _ptr(res.dist, _u32p)
        rs.hops = _ptr(res.hops, _u16p)
        rs.first_parent = _ptr(res.first_parent, _u32p)
        rs.n_parents = _ptr(res.n_parents, _u16p)
        rs.nh_mask = _ptr(res.nh_mask, _u64p)
        rs.nh_words = nh_words
        rs.job_status = _ptr(res.job_status, _u32p)
        rc = self.lib.hspf_run_batch(self.handle, graph.handle, C.byref(js), C.byref(rs), 0)
        res.status = self._check(rc, allow=(HSPF_E_JOB_STATUS,))
        del keep
        return res

    def run16(self, graph: Graph, roots, overrides=None, planes=("dist", "hops", "first_parent", "n_parents", "nh_mask")):
        """Host-pointer call with 16-bit planes (hspf_run_batch16); planes not listed are skipped (NULL)."""
        js, keep = make_jobs(roots, overrides)
        n, V = js.n_jobs, graph.csr.n_vertices
        arr = {k: np.empty((n, V), np.uint16) for k in planes}
        status = np.zeros(n, np.uint32)
        rs = Result16Struct()
        for k in ("dist", "hops", "first_parent", "n_parents", "nh_mask"):
            setattr(rs, k, _ptr(arr.get(k), _u16p))
        rs.job_status = _ptr(status, _u32p)
        rc = self.lib.hspf_run_batch16(self.handle, graph.handle, C.byref(js), C.byref(rs), 0)
        rc = self._check(rc, allow=(HSPF_E_JOB_STATUS,))
        del keep
        arr["job_status"] = status
        arr["status"] = rc
        return arr

    def run_device16(self, graph: Graph, jobs: JobsStruct, rs: "Result16Struct", sync: bool = True):
        """Device-pointer call with 16-bit planes."""
        self._check(self.lib.hspf_run_batch16_async(self.handle, graph.handle, C.byref(jobs), C.byref(rs)))
        if sync:
            self._check(self.lib.hspf_sync(self.handle))

    def graph_info(self, graph: Graph) -> dict:
        info = (C.c_uint32 * 8)()
        self._check(self.lib.hspf_graph_info(graph.handle, info))
        return {"fast_path": bool(info[0]), "fwd_quads": info[1], "in_quads": info[2], "bucket_shift": info[3],
                "V": info[4], "E": info[5], "max_indeg": info[6]}

    def run_device(self, graph: Graph, jobs: JobsStruct, rs: ResultStruct, sync: bool = True):
        """Device-pointer call (inputs/outputs already resident in HBM)."""
        self._check(self.lib.hspf_run_batch_async(self.handle, graph.handle, C.byref(jobs), C.byref(rs)))
        if sync:
            self._check(self.lib.hspf_sync(self.handle))

    def sync(self):
        self._check(self.lib.hspf_sync(self.handle))

    def update_costs(self, graph: "Graph", edges, costs):
        """hspf_graph_update_costs: permanent cost change of existing edges, patched in place on the device."""
        e = np.ascontiguousarray(edges, np.uint32)
        c = np.ascontiguousarray(costs, np.uint32)
        assert e.shape == c.shape
        self.lib.hspf_graph_update_costs.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        self._check(self.lib.hspf_graph_update_costs(self.handle, graph.handle, len(e), e.ctypes.data, c.ctypes.data))

    def set_peer_slots(self, deltas):
        """Fused exchange: the next 16-bit launches also store dist / hops / nh_mask / status into the
        peers' copies of this rank's slot (hspf_xchg_peer_deltas); [] switches it off."""
        self.lib.hspf_ctx_set_peer_slots.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_int64)]
        arr = (C.c_int64 * max(len(deltas), 1))(*deltas)
        self._check(self.lib.hspf_ctx_set_peer_slots(self.handle, len(deltas), arr))

    @contextmanager
    def path(self, name: str):
        """Test aid: the batches of the `with` block run on one kernel path (hspf_debug_set_path):
        "auto" (the default), "general" or "general_kahn"."""
        self._check(self.lib.hspf_debug_set_path(self.handle, PATHS[name]))
        try:
            yield
        finally:
            self._check(self.lib.hspf_debug_set_path(self.handle, PATHS["auto"]))

    def reserve_sms(self, n_sms: int):
        self._check(self.lib.hspf_ctx_reserve_sms(self.handle, n_sms))

    @property
    def stream(self) -> int:
        return int(self.lib.hspf_stream(self.handle) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.hspf_launch_count(self.handle))


@dataclass
class QuadImage:
    """Host copy of the quad-space graph image (csrc/quad_layout.h), for tests."""
    eligible: bool
    NQ: int = 0
    NIQ: int = 0
    shift: int = 0
    max_ichain: int = 1
    max_atoms: int = 0
    fq: np.ndarray | None = None       # [NQ, 4]
    fcont: np.ndarray | None = None    # [NQ / 32]
    slot_of: np.ndarray | None = None  # [V]
    vert_of: np.ndarray | None = None  # [NQ]
    iq: np.ndarray | None = None       # [NIQ, 4]
    imeta: np.ndarray | None = None    # [NIQ, 2]
    fpos: np.ndarray | None = None     # [E]
    ipos: np.ndarray | None = None     # [E]


def quad_image(csr: Csr) -> QuadImage:
    """Build the quad-space image on the host (no CUDA call)."""
    lib = load_library()
    s = csr.as_struct()
    hdr = (C.c_uint32 * 8)()
    nul32, nul16 = C.cast(None, _u32p), C.cast(None, _u16p)
    rc = lib.hspf_debug_quad_image(C.byref(s), hdr, nul32, nul32, nul16, nul16, nul32, nul32, nul32, nul32)
    if rc != HSPF_OK:
        raise HspfError(rc, "hspf_debug_quad_image")
    if not hdr[0]:
        return QuadImage(False)
    NQ, NIQ, V, E = hdr[1], hdr[2], csr.n_vertices, csr.n_edges
    q = QuadImage(True, NQ, NIQ, hdr[3], hdr[4], hdr[5],
                  np.zeros((NQ, 4), np.uint32), np.zeros(NQ // 32, np.uint32), np.zeros(V, np.uint16),
                  np.zeros(NQ, np.uint16), np.zeros((NIQ, 4), np.uint32), np.zeros((NIQ, 2), np.uint32),
                  np.zeros(max(E, 1), np.uint32), np.zeros(max(E, 1), np.uint32))
    rc = lib.hspf_debug_quad_image(C.byref(s), hdr, _ptr(q.fq, _u32p), _ptr(q.fcont, _u32p), _ptr(q.slot_of, _u16p),
                                   _ptr(q.vert_of, _u16p), _ptr(q.iq, _u32p), _ptr(q.imeta, _u32p),
                                   _ptr(q.fpos, _u32p), _ptr(q.ipos, _u32p))
    if rc != HSPF_OK:
        raise HspfError(rc, "hspf_debug_quad_image")
    q.fpos, q.ipos = q.fpos[:E], q.ipos[:E]
    return q


def atom_decode(csr: Csr, root: int, atom: int):
    lib = load_library()
    s = csr.as_struct()
    t, e = C.c_uint32(), C.c_uint32()
    rc = lib.hspf_atom_decode(C.byref(s), root, atom, C.byref(t), C.byref(e))
    if rc != HSPF_OK:
        raise HspfError(rc, "atom out of range")
    return t.value, e.value


def atom_count(csr: Csr, root: int) -> int:
    lib = load_library()
    s = csr.as_struct()
    n = C.c_uint32()
    rc = lib.hspf_atom_count(C.byref(s), root, C.byref(n))
    if rc != HSPF_OK:
        raise HspfError(rc, "bad root")
    return n.value
