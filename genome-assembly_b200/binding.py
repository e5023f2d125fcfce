"""ctypes mirror of include/gbin.h (libgbin.so).  No computation happens in Python and there is no
fallback: if the shared library is missing, or the machine has no CUDA device, calls raise."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgbin.so")

GBIN_OK = 0
GBIN_E_INVALID_CONFIG = -1
GBIN_E_CUDA = -2
GBIN_E_NOMEM = -3
GBIN_E_NON_ACGT = -4
GBIN_E_STATE = -5
GBIN_E_TOO_LARGE = -6
GBIN_E_INVALID_ARG = -7
GBIN_E_IO = -8


class GbinError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"gbin error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("kmer_size", C.c_int32), ("mmer_size", C.c_int32), ("abundance_cutoff", C.c_int32), ("device", C.c_int32)]


class CTable(C.Structure):
    _fields_ = [("kmer_size", C.c_int32), ("mmer_size", C.c_int32), ("abundance_cutoff", C.c_int32), ("kmer_words", C.c_int32),
                ("on_device", C.c_int32), ("ctx_owned", C.c_int32),
                ("n_instances", C.c_uint64), ("n_distinct", C.c_uint64), ("n_buckets", C.c_uint64), ("n_kmers", C.c_uint64),
                ("n_ids", C.c_uint64),
                ("mmer_codes", C.c_void_p), ("mmer_kmer_off", C.c_void_p), ("kmer_codes", C.c_void_p),
                ("kmer_id_off", C.c_void_p), ("read_ids", C.c_void_p)]


class CExpanded(C.Structure):
    """gbin_expanded: the list of lists expand_read_id_list builds (binning.c:857-888), in CSR form."""
    _fields_ = [("kmer_size", C.c_int32), ("on_device", C.c_int32), ("n_lists", C.c_uint64), ("n_ids", C.c_uint64),
                ("list_off", C.c_void_p), ("ids", C.c_void_p)]


class CReads(C.Structure):
    _fields_ = [("data", C.c_void_p), ("data_bytes", C.c_uint64), ("n_reads", C.c_uint64), ("stride", C.c_uint64),
                ("read_len", C.c_uint32), ("id_base", C.c_int32), ("starts", C.c_void_p), ("lens", C.c_void_p),
                ("read_ids", C.c_void_p), ("max_read_len", C.c_uint32), ("reserved", C.c_uint32)]


class Timings(C.Structure):
    _fields_ = [("h2d_ms", C.c_float), ("scan_ms", C.c_float), ("sort_ms", C.c_float), ("group_ms", C.c_float),
                ("d2h_ms", C.c_float), ("total_ms", C.c_float), ("kernel_launches", C.c_uint32), ("sort_passes", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class KernelProfile(C.Structure):
    _fields_ = [("ms", C.c_float * 12), ("launches", C.c_uint32 * 12)]


# every symbol include/gbin.h declares (tests check that the library exports all of them)
EXPORTS = [
    "gbin_strerror", "gbin_last_error", "gbin_version", "gbin_create", "gbin_destroy", "gbin_get_config",
    "gbin_bin_reads_host", "gbin_table_clone", "gbin_table_free", "gbin_pinned_alloc", "gbin_pinned_free",
    "gbin_bin_reads_device", "gbin_table_to_host", "gbin_table_to_pinned", "gbin_get_timings", "gbin_record_bytes",
    "gbin_set_kernel_profiling", "gbin_get_kernel_profile", "gbin_kernel_kind_name", "gbin_max_read_len", "gbin_multi_create", "gbin_multi_destroy", "gbin_multi_devices", "gbin_multi_context", "gbin_multi_last_error", "gbin_multi_bin_reads_host",
    "gbin_bin_reads_host_part", "gbin_bin_reads_device_part", "gbin_plan_parts", "gbin_table_digest", "gbin_set_pipeline", "gbin_set_tuning", "gbin_donate_scratch", "gbin_get_pipeline_info", "gbin_get_run_stats",
    "gbin_count_instances_device", "gbin_scan_reads_device", "gbin_partition_records_device",
    "gbin_group_records_device", "gbin_owner_of", "gbin_xchg_create", "gbin_xchg_attach", "gbin_xchg_exchange_skr", "gbin_xchg_detach", "gbin_xchg_destroy", "gbin_skr_record_bytes", "gbin_scan_skr_device", "gbin_partition_skr_device", "gbin_group_skr_device",
    "gbin_split_reads_device", "gbin_copy_to_host", "gbin_bin_file_host", "gbin_read_file_fgets", "gbin_table_dump", "gbin_table_dump_reference_format", "gbin_table_dump_expanded_format",
    "gbin_expand_read_ids_device", "gbin_expanded_to_host", "gbin_expanded_free", "gbin_table_dump_expanded_lists",
    "getval", "getbp", "getscore", "process_read", "prune_data", "gbin_ref_configure", "gbin_ref_last_status",
    "gbin_ref_reset", "gbin_table_to_zhash", "gbin_zhash_release",
]

_lib = None


def load_library() -> C.CDLL:
    """Loads libgbin.so (built in-tree by `make -C genome-assembly_b200` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `make -C genome-assembly_b200` "
                          "(there is no CPU or PyTorch fallback for the binning path)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
    L.gbin_strerror.restype = C.c_char_p
    L.gbin_strerror.argtypes = [C.c_int]
    L.gbin_last_error.restype = C.c_char_p
    L.gbin_last_error.argtypes = [vp]
    L.gbin_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.gbin_destroy.argtypes = [vp]
    L.gbin_destroy.restype = None
    L.gbin_get_config.argtypes = [vp, C.POINTER(Config)]
    L.gbin_bin_reads_host.argtypes = [vp, C.POINTER(CReads), C.POINTER(CTable)]
    L.gbin_bin_reads_device.argtypes = [vp, C.POINTER(CReads), vp, C.POINTER(CTable)]
    L.gbin_bin_reads_host_part.argtypes = [vp, C.POINTER(CReads), u32, u32, C.POINTER(CTable)]
    L.gbin_bin_reads_device_part.argtypes = [vp, C.POINTER(CReads), u32, u32, vp, C.POINTER(CTable)]
    L.gbin_plan_parts.argtypes = [vp, u64, C.POINTER(u32)]
    L.gbin_table_to_host.argtypes = [vp, C.POINTER(CTable), C.POINTER(CTable)]
    L.gbin_table_to_pinned.argtypes = [vp, C.POINTER(CTable), vp, C.POINTER(CTable)]
    L.gbin_table_clone.argtypes = [C.POINTER(CTable), C.POINTER(CTable)]
    L.gbin_table_free.argtypes = [C.POINTER(CTable)]
    L.gbin_table_free.restype = None
    L.gbin_pinned_alloc.argtypes = [C.c_size_t]
    L.gbin_pinned_alloc.restype = vp
    L.gbin_pinned_free.argtypes = [vp]
    L.gbin_pinned_free.restype = None
    L.gbin_get_timings.argtypes = [vp, C.POINTER(Timings)]
    L.gbin_get_run_stats.argtypes = [vp, C.POINTER(u64 * 6)]
    L.gbin_set_pipeline.argtypes = [vp, C.c_int]
    L.gbin_table_digest.argtypes = [vp, C.POINTER(CTable), vp, C.POINTER(u64)]
    L.gbin_set_tuning.argtypes = [vp, C.c_char_p, C.c_int]
    L.gbin_donate_scratch.argtypes = [vp, vp, C.c_uint64]
    L.gbin_get_pipeline_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_uint32)]
    L.gbin_set_kernel_profiling.argtypes = [vp, C.c_int]
    L.gbin_get_kernel_profile.argtypes = [vp, C.POINTER(KernelProfile)]
    L.gbin_kernel_kind_name.argtypes = [C.c_int]
    L.gbin_kernel_kind_name.restype = C.c_char_p
    L.gbin_record_bytes.argtypes = [vp]
    L.gbin_record_bytes.restype = u32
    L.gbin_max_read_len.restype = u32
    L.gbin_max_read_len.argtypes = []
    L.gbin_count_instances_device.argtypes = [vp, C.POINTER(CReads), vp, C.POINTER(u64)]
    L.gbin_scan_reads_device.argtypes = [vp, C.POINTER(CReads), u32, vp, u64, vp, C.POINTER(u64)]
    L.gbin_partition_records_device.argtypes = [vp, vp, u64, u32, vp, vp, C.POINTER(u64)]
    L.gbin_group_records_device.argtypes = [vp, vp, u64, vp, i32, vp, C.POINTER(CTable)]
    L.gbin_skr_record_bytes.argtypes = [vp]
    L.gbin_skr_record_bytes.restype = u32
    L.gbin_scan_skr_device.argtypes = [vp, C.POINTER(CReads), u32, vp, u64, vp, C.POINTER(u64), C.POINTER(u64)]
    L.gbin_partition_skr_device.argtypes = [vp, vp, u64, u32, vp, vp, C.POINTER(u64)]
    L.gbin_group_skr_device.argtypes = [vp, vp, u64, vp, i32, vp, C.POINTER(CTable), C.POINTER(C.c_int)]
    L.gbin_owner_of.argtypes = [u32, u32]
    L.gbin_owner_of.restype = u32
    L.gbin_xchg_create.argtypes = [vp, u32, u32, u64, vp]
    L.gbin_xchg_attach.argtypes = [vp, vp]
    L.gbin_xchg_exchange_skr.argtypes = [vp, vp, u64, vp, C.POINTER(vp), C.POINTER(u64), C.POINTER(u64)]
    L.gbin_xchg_destroy.argtypes = [vp]
    L.gbin_xchg_destroy.restype = None
    L.gbin_xchg_detach.argtypes = [vp]
    L.gbin_xchg_detach.restype = None
    L.gbin_split_reads_device.argtypes = [vp, vp, u64, C.c_int, vp, C.POINTER(CReads)]
    L.gbin_copy_to_host.argtypes = [vp, vp, vp, u64]
    L.gbin_bin_file_host.argtypes = [vp, C.c_char_p, C.c_int, C.POINTER(CTable)]
    L.gbin_read_file_fgets.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp), C.POINTER(u64), C.POINTER(vp), C.POINTER(vp),
                                       C.POINTER(u64)]
    L.gbin_table_dump.argtypes = [C.POINTER(CTable), C.c_char_p]
    L.gbin_table_dump_reference_format.argtypes = [C.POINTER(CTable), C.c_char_p]
    L.gbin_table_dump_expanded_format.argtypes = [C.POINTER(CTable), C.c_char_p]
    L.gbin_expand_read_ids_device.argtypes = [C.c_void_p, C.POINTER(CTable), C.c_void_p, C.POINTER(CExpanded)]
    L.gbin_expanded_to_host.argtypes = [C.c_void_p, C.POINTER(CExpanded), C.POINTER(CExpanded)]
    L.gbin_expanded_free.argtypes = [C.POINTER(CExpanded)]
    L.gbin_expanded_free.restype = None
    L.gbin_table_dump_expanded_lists.argtypes = [C.POINTER(CTable), C.POINTER(CExpanded), C.c_char_p]
    L.getval.argtypes = [C.c_char]
    L.getval.restype = C.c_int
    L.getbp.argtypes = [C.c_int]
    L.getbp.restype = C.c_char
    L.getscore.argtypes = [C.c_char_p]
    L.getscore.restype = C.c_int
    L.process_read.argtypes = [vp, C.c_char_p, C.c_int]
    L.process_read.restype = vp
    L.prune_data.argtypes = [vp]
    L.prune_data.restype = vp
    L.gbin_ref_configure.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    L.gbin_ref_last_status.restype = C.c_int
    L.gbin_ref_reset.argtypes = [vp]
    L.gbin_ref_reset.restype = None
    L.gbin_table_to_zhash.argtypes = [C.POINTER(CTable), vp]
    L.gbin_zhash_release.argtypes = [vp]
    L.gbin_zhash_release.restype = None
    _lib = L
    return L


@dataclass
class HostTable:
    """The pruned mmer -> kmer -> read-id table as numpy arrays (copies; canonical order)."""
    K: int
    M: int
    cutoff: int
    kw: int
    n_instances: int
    n_distinct: int
    mmer_codes: np.ndarray
    mmer_kmer_off: np.ndarray
    kmer_codes: np.ndarray
    kmer_id_off: np.ndarray
    read_ids: np.ndarray

    @property
    def n_buckets(self):
        return len(self.mmer_codes)

    @property
    def n_kmers(self):
        return len(self.kmer_id_off) - 1

    @property
    def n_ids(self):
        return len(self.read_ids)


def _np_from(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=n).copy()


def host_table_from_c(t: CTable) -> HostTable:
    assert not t.on_device
    return HostTable(K=t.kmer_size, M=t.mmer_size, cutoff=t.abundance_cutoff, kw=t.kmer_words,
                     n_instances=int(t.n_instances), n_distinct=int(t.n_distinct),
                     mmer_codes=_np_from(t.mmer_codes, t.n_buckets, np.uint32),
                     mmer_kmer_off=_np_from(t.mmer_kmer_off, t.n_buckets + 1, np.uint64),
                     kmer_codes=_np_from(t.kmer_codes, t.n_kmers * t.kmer_words, np.uint64),
                     kmer_id_off=_np_from(t.kmer_id_off, t.n_kmers + 1, np.uint64),
                     read_ids=_np_from(t.read_ids, t.n_ids, np.int32))


def owner_of(mmer_codes, parts: int) -> np.ndarray:
    """gbin_owner_of for an array of m-mer codes: which of `parts` GPUs owns each bucket."""
    m = np.asarray(mmer_codes).astype(np.uint64)
    return ((((m * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) * np.uint64(parts)) >> np.uint64(32)).astype(np.int64)


CUDA_STREAM_LEGACY = 1  # cudaStreamLegacy: explicit handle of the legacy default stream


def stream_handle(torch_stream) -> int:
    """cudaStream_t to hand to the C ABI for a torch stream.  torch's default stream has handle 0, which
    the C ABI reads as "use the context's own stream"; map it to cudaStreamLegacy so that work is
    ordered with whatever torch enqueued on its default stream."""
    h = int(torch_stream.cuda_stream)
    return h if h else CUDA_STREAM_LEGACY


def _ptr(x):
    """Raw address of a numpy array / torch tensor / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    raise TypeError(type(x))


class Binner:
    """One context per GPU (gbin_ctx): K, M and the cutoff are the runtime form of binning.c:10-12."""

    def __init__(self, k: int = 31, m: int = 4, cutoff: int = 1, device: int = 0, pipeline: int | None = None):
        self.lib = load_library()
        self.cfg = Config(k, m, cutoff, device)
        h = C.c_void_p()
        rc = self.lib.gbin_create(C.byref(self.cfg), C.byref(h))
        if rc != GBIN_OK:
            raise GbinError(rc, self.lib.gbin_strerror(rc).decode())
        self.h = h
        self.k, self.m, self.cutoff, self.device = k, m, cutoff, device
        if pipeline is not None:
            self.set_pipeline(pipeline)

    def close(self):
        if getattr(self, "h", None):
            self.lib.gbin_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != GBIN_OK:
            raise GbinError(rc, f"{self.lib.gbin_strerror(rc).decode()}: {self.lib.gbin_last_error(self.h).decode()}")

    @property
    def record_bytes(self) -> int:
        return int(self.lib.gbin_record_bytes(self.h))

    def timings(self) -> dict:
        t = Timings()
        self.lib.gbin_get_timings(self.h, C.byref(t))
        return t.as_dict()

    def set_pipeline(self, pipeline: int):
        self._check(self.lib.gbin_set_pipeline(self.h, pipeline))

    def table_digest(self, table: CTable, stream=None) -> int:
        """Order-independent 64-bit digest of a device or host table (gbin_table_digest)."""
        d = C.c_uint64()
        self._check(self.lib.gbin_table_digest(self.h, C.byref(table), stream, C.byref(d)))
        return int(d.value)

    def expand_read_ids_device(self, dev_table: CTable, stream=None) -> CExpanded:
        """expand_read_id_list on the device: K copies of every surviving k-mer's id list (device memory of the context)."""
        x = CExpanded()
        self._check(self.lib.gbin_expand_read_ids_device(self.h, C.byref(dev_table), stream, C.byref(x)))
        return x

    def expanded_to_host(self, dev: CExpanded) -> CExpanded:
        h = CExpanded()
        self._check(self.lib.gbin_expanded_to_host(self.h, C.byref(dev), C.byref(h)))
        return h

    def donate_scratch(self, d_buf, nbytes: int):
        """Lends device memory to the next grouping call (gbin_donate_scratch); keep `d_buf` alive until that call has returned."""
        self._check(self.lib.gbin_donate_scratch(self.h, _ptr(d_buf), int(nbytes)))

    def set_tuning(self, name: str, value: int):
        self._check(self.lib.gbin_set_tuning(self.h, name.encode(), int(value)))

    def pipeline_info(self) -> dict:
        a, b, c = C.c_int(), C.c_int(), C.c_uint32()
        self._check(self.lib.gbin_get_pipeline_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return {"configured": a.value, "last_used": b.value, "fallbacks": c.value}

    def run_stats(self) -> dict:
        a = (C.c_uint64 * 6)()
        self._check(self.lib.gbin_get_run_stats(self.h, C.byref(a)))
        return {"n_super_kmers": int(a[0]), "n_mmer_runs": int(a[1]), "n_units": int(a[2]), "n_lsd_kmers": int(a[3]),
                "key_nc": int(a[4]) & 0xffffffff, "key_h": int(a[4]) >> 32, "n_passes": int(a[5]) & 0xffffffff}

    def set_kernel_profiling(self, enable: bool):
        self._check(self.lib.gbin_set_kernel_profiling(self.h, int(enable)))

    def kernel_profile(self) -> dict:
        """{kernel class: {"ms": accumulated device ms, "launches": n}} since profiling was enabled."""
        p = KernelProfile()
        self._check(self.lib.gbin_get_kernel_profile(self.h, C.byref(p)))
        out = {}
        for i in range(12):
            name = self.lib.gbin_kernel_kind_name(i).decode()
            if name:
                out[name] = {"ms": float(p.ms[i]), "launches": int(p.launches[i])}
        return out

    @staticmethod
    def _reads(data, data_bytes, n_reads, stride=0, read_len=0, starts=None, lens=None, read_ids=None, id_base=0, max_read_len=0):
        return CReads(_ptr(data), data_bytes, n_reads, stride, read_len, id_base, _ptr(starts), _ptr(lens), _ptr(read_ids),
                      max_read_len, 0)

    # ---- host buffers in, host table out (H2D + pipeline + D2H)
    def bin_host_raw(self, reads: CReads) -> CTable:
        """Returns the ctx-owned pinned table (valid until the next call) without copying it."""
        t = CTable()
        self._check(self.lib.gbin_bin_reads_host(self.h, C.byref(reads), C.byref(t)))
        return t

    @staticmethod
    def _host_reads(data, n_reads, stride, read_len, starts, lens, read_ids, id_base):
        """-> (CReads over numpy copies of the arguments, the arrays it points into: keep them alive for the call)."""
        if isinstance(data, (bytes, bytearray)):
            data = np.frombuffer(data, dtype=np.uint8)
        data = np.ascontiguousarray(data, dtype=np.uint8)
        keep = [data]
        if starts is not None:
            starts = np.ascontiguousarray(starts, dtype=np.uint64)
            lens = np.ascontiguousarray(lens, dtype=np.uint32)
            keep += [starts, lens]
        if read_ids is not None:
            read_ids = np.ascontiguousarray(read_ids, dtype=np.int32)
            keep.append(read_ids)
        return Binner._reads(data, data.size, n_reads, stride, read_len, starts, lens, read_ids, id_base), keep

    def bin_host(self, data, n_reads, *, stride=0, read_len=0, starts=None, lens=None, read_ids=None, id_base=0) -> HostTable:
        rd, _keep = self._host_reads(data, n_reads, stride, read_len, starts, lens, read_ids, id_base)
        return host_table_from_c(self.bin_host_raw(rd))

    # ---- read sets larger than one device: part `part` of `n_parts` owner parts of the table per call
    def bin_host_part_raw(self, reads: CReads, part: int, n_parts: int) -> CTable:
        """gbin_bin_reads_host_part: the ctx-owned pinned table of the part (valid until the next call) without copying it."""
        t = CTable()
        self._check(self.lib.gbin_bin_reads_host_part(self.h, C.byref(reads), part, n_parts, C.byref(t)))
        return t

    def bin_host_part(self, data, n_reads, part: int, n_parts: int, *, stride=0, read_len=0, starts=None, lens=None, read_ids=None,
                      id_base=0) -> HostTable:
        rd, _keep = self._host_reads(data, n_reads, stride, read_len, starts, lens, read_ids, id_base)
        return host_table_from_c(self.bin_host_part_raw(rd, part, n_parts))

    def bin_device_part_raw(self, reads: CReads, part: int, n_parts: int, stream: int | None = None) -> CTable:
        """gbin_bin_reads_device_part: reads in device memory, the part's table in the context's device memory."""
        t = CTable()
        self._check(self.lib.gbin_bin_reads_device_part(self.h, C.byref(reads), part, n_parts, stream, C.byref(t)))
        return t

    def plan_parts(self, n_instances: int) -> int:
        """gbin_plan_parts: the smallest number of parts whose one part fits the device's free memory now."""
        p = C.c_uint32()
        self._check(self.lib.gbin_plan_parts(self.h, int(n_instances), C.byref(p)))
        return int(p.value)

    # ---- device buffers in, device table out
    def bin_device_raw(self, reads: CReads, stream: int | None = None) -> CTable:
        t = CTable()
        self._check(self.lib.gbin_bin_reads_device(self.h, C.byref(reads), stream, C.byref(t)))
        return t

    def table_to_host(self, dev: CTable) -> HostTable:
        h = CTable()
        self._check(self.lib.gbin_table_to_host(self.h, C.byref(dev), C.byref(h)))
        try:
            return host_table_from_c(h)
        finally:
            self.lib.gbin_table_free(C.byref(h))

    def table_to_pinned_raw(self, dev: CTable, stream=None) -> CTable:
        """Device table -> the context's pinned arena (valid until the next host-table call); no numpy copies."""
        h = CTable()
        self._check(self.lib.gbin_table_to_pinned(self.h, C.byref(dev), stream, C.byref(h)))
        return h

    # ---- main's read loop on the device
    def split_reads_device(self, d_data, data_bytes: int, read_length_define: int, stream=None) -> CReads:
        """fgets-style split of a file image in device memory -> ragged CReads with device pointers (context-owned)."""
        rd = CReads()
        self._check(self.lib.gbin_split_reads_device(self.h, _ptr(d_data), data_bytes, read_length_define, stream, C.byref(rd)))
        return rd

    def device_array(self, dev_ptr, n: int, dtype) -> np.ndarray:
        """Host copy of n elements at a device address (context-owned device arrays)."""
        out = np.zeros(n, dtype=dtype)
        if n:
            self._check(self.lib.gbin_copy_to_host(self.h, out.ctypes.data, int(dev_ptr), out.nbytes))
        return out

    def bin_file_host(self, path: str, read_length_define: int) -> HostTable:
        """File -> pruned table: the file is split into reads on the device exactly as main's fgets loop does."""
        t = CTable()
        self._check(self.lib.gbin_bin_file_host(self.h, path.encode(), read_length_define, C.byref(t)))
        return host_table_from_c(t)

    # ---- staged device entry points
    def count_instances_device(self, reads: CReads, stream=None) -> int:
        n = C.c_uint64()
        self._check(self.lib.gbin_count_instances_device(self.h, C.byref(reads), stream, C.byref(n)))
        return int(n.value)

    def scan_device(self, reads: CReads, arrival_base: int, d_records, capacity: int, stream=None) -> int:
        n = C.c_uint64()
        self._check(self.lib.gbin_scan_reads_device(self.h, C.byref(reads), arrival_base, _ptr(d_records), capacity, stream, C.byref(n)))
        return int(n.value)

    def partition_device(self, d_records, n: int, n_parts: int, d_out, stream=None) -> list[int]:
        counts = (C.c_uint64 * n_parts)()
        self._check(self.lib.gbin_partition_records_device(self.h, _ptr(d_records), n, n_parts, _ptr(d_out), stream, counts))
        return [int(c) for c in counts]

    # ---- staged entry points, super-k-mer form
    @property
    def skr_record_bytes(self) -> int:
        return int(self.lib.gbin_skr_record_bytes(self.h))

    def scan_skr_device(self, reads: CReads, arrival_base: int, d_skr, capacity: int, stream=None):
        """-> (n_records, n_instances)"""
        n, ni = C.c_uint64(), C.c_uint64()
        self._check(self.lib.gbin_scan_skr_device(self.h, C.byref(reads), arrival_base, _ptr(d_skr), capacity, stream, C.byref(n), C.byref(ni)))
        return int(n.value), int(ni.value)

    def partition_skr_device(self, d_skr, n: int, n_parts: int, d_out, stream=None) -> list[int]:
        counts = (C.c_uint64 * n_parts)()
        self._check(self.lib.gbin_partition_skr_device(self.h, _ptr(d_skr), n, n_parts, _ptr(d_out), stream, counts))
        return [int(c) for c in counts]

    def group_skr_device(self, d_skr, n_skr: int, d_ids_by_arrival=None, id_base: int = 0, stream=None) -> CTable:
        t = CTable()
        fb = C.c_int()
        self._check(self.lib.gbin_group_skr_device(self.h, _ptr(d_skr), n_skr, _ptr(d_ids_by_arrival), id_base, stream, C.byref(t), C.byref(fb)))
        return t

    # ---- owner exchange over peer memory (collective over the ranks whose contexts were attached to each other)
    XCHG_HANDLE_BYTES = 192

    def xchg_create(self, rank: int, world: int, capacity_records: int) -> bytes:
        buf = C.create_string_buffer(self.XCHG_HANDLE_BYTES)
        self._check(self.lib.gbin_xchg_create(self.h, rank, world, capacity_records, buf))
        return buf.raw

    def xchg_attach(self, all_handles: bytes):
        self._check(self.lib.gbin_xchg_attach(self.h, C.c_char_p(all_handles)))

    def xchg_exchange_skr(self, d_skr, n: int, world: int, stream=None):
        """-> (device address of this rank's receive buffer, records received, records sent per owner)"""
        recv, n_in = C.c_void_p(), C.c_uint64()
        sent = (C.c_uint64 * 16)()
        self._check(self.lib.gbin_xchg_exchange_skr(self.h, _ptr(d_skr), n, stream, C.byref(recv), C.byref(n_in), sent))
        return int(recv.value or 0), int(n_in.value), [int(sent[i]) for i in range(world)]

    def xchg_detach(self):
        self.lib.gbin_xchg_detach(self.h)

    def xchg_destroy(self):
        self.lib.gbin_xchg_destroy(self.h)

    def group_device(self, d_records, n: int, d_ids_by_arrival=None, id_base: int = 0, stream=None) -> CTable:
        t = CTable()
        self._check(self.lib.gbin_group_records_device(self.h, _ptr(d_records), n, _ptr(d_ids_by_arrival), id_base, stream, C.byref(t)))
        return t


def read_file_fgets(path: str, read_length_define: int):
    """main's read loop (binning.c:1154-1166) -> (data bytes, starts u64[n], lens u32[n])."""
    L = load_library()
    data, starts, lens = C.c_void_p(), C.c_void_p(), C.c_void_p()
    nbytes, n = C.c_uint64(), C.c_uint64()
    rc = L.gbin_read_file_fgets(path.encode(), read_length_define, C.byref(data), C.byref(nbytes), C.byref(starts), C.byref(lens),
                                C.byref(n))
    if rc != GBIN_OK:
        raise GbinError(rc, L.gbin_strerror(rc).decode())
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    try:
        return (_np_from(data.value, nbytes.value, np.uint8), _np_from(starts.value, n.value, np.uint64),
                _np_from(lens.value, n.value, np.uint32))
    finally:
        for p in (data, starts, lens):
            libc.free(p)
