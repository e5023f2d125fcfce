"""The checks every entry point that takes a reads descriptor makes before it copies or launches anything, and valid host layouts
that are unusual.  Every malformed descriptor must return its code from each entry point it applies to (the multi-GPU call at G = 1
through ctypes), and the same contexts must then still bin a valid batch to the oracle's table.  Every buffer a malformed descriptor
points into is larger than the data_bytes it claims, so that a missing check could only read memory the test owns."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from genome_assembly_b200 import binding as B
from test_gpu_parts import check_parts
from test_gpu_sharded import assert_tables_equal, caller_ids, get_input, oracle_table, oracle_tuples, torch_cuda

pytestmark = pytest.mark.gpu

PAD = 1 << 16  # bytes behind what a descriptor claims
HOST_ENTRIES = ("host", "host_part", "multi")
ALL_ENTRIES = ("host", "device", "host_part", "device_part", "count", "scan_reads", "scan_skr", "multi")


def multi_lib():
    L = B.load_library()
    L.gbin_multi_create.argtypes = [C.POINTER(B.Config), C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    L.gbin_multi_bin_reads_host.argtypes = [C.c_void_p, C.POINTER(B.CReads), C.POINTER(B.CTable)]
    L.gbin_multi_destroy.argtypes = [C.c_void_p]
    L.gbin_multi_destroy.restype = None
    L.gbin_multi_last_error.argtypes = [C.c_void_p]
    L.gbin_multi_last_error.restype = C.c_char_p
    return L


class Multi:
    """gbin_multi over device 0 only (G = 1)."""

    def __init__(self, K, M, cutoff):
        self.lib = multi_lib()
        self.h = C.c_void_p()
        rc = self.lib.gbin_multi_create(C.byref(B.Config(K, M, cutoff, 0)), (C.c_int * 1)(0), 1, C.byref(self.h))
        assert rc == B.GBIN_OK, rc

    def bin_raw(self, rd):
        """-> (return code, the host table of the one GPU)."""
        t = (B.CTable * 1)()
        return self.lib.gbin_multi_bin_reads_host(self.h, C.byref(rd), t), t[0]

    def close(self):
        if self.h:
            self.lib.gbin_multi_destroy(self.h)
            self.h = None


# ---------------------------------------------------------------- malformed descriptors

def _ragged(n=10, read_len=100):
    return np.arange(n, dtype=np.uint64) * read_len, np.full(n, read_len, np.uint32)


def _edit(a, i, v):
    a = a.copy()
    a[i] = v
    return a


S, LN = _ragged()
# name -> (descriptor fields, expected code, entry points it applies to).  Fields: n, data_bytes, stride, read_len, starts, lens,
# max_read_len, and null_data for a NULL data pointer.  Ragged reads in device memory are not checked against data_bytes.
CASES = {
    "data_null": (dict(n=10, data_bytes=1000, stride=100, read_len=100, null_data=True), B.GBIN_E_INVALID_ARG, ALL_ENTRIES),
    "too_many_reads": (dict(n=1 << 32, data_bytes=1000, stride=100, read_len=100), B.GBIN_E_TOO_LARGE, ALL_ENTRIES),
    "host_without_data_bytes": (dict(n=10, data_bytes=0, stride=100, read_len=100), B.GBIN_E_INVALID_ARG, HOST_ENTRIES),
    "stride_below_read_len": (dict(n=10, data_bytes=1000, stride=50, read_len=100), B.GBIN_E_INVALID_ARG, ALL_ENTRIES),
    "fixed_past_data_bytes": (dict(n=10, data_bytes=950, stride=100, read_len=100), B.GBIN_E_INVALID_ARG, ALL_ENTRIES),
    # (n - 1) * stride wraps to 0 modulo 2^64: the span must be checked without overflow
    "fixed_span_wraps": (dict(n=5, data_bytes=1000, stride=1 << 62, read_len=100), B.GBIN_E_INVALID_ARG, ALL_ENTRIES),
    "ragged_without_lens": (dict(n=10, data_bytes=1000, starts=S), B.GBIN_E_INVALID_ARG, ALL_ENTRIES),
    "ragged_past_data_bytes": (dict(n=10, data_bytes=1000, starts=_edit(S, 9, 950), lens=LN), B.GBIN_E_INVALID_ARG, HOST_ENTRIES),
    "ragged_past_data_bytes_with_max": (dict(n=10, data_bytes=1000, starts=_edit(S, 9, 950), lens=LN, max_read_len=150),
                                        B.GBIN_E_INVALID_ARG, HOST_ENTRIES),
    # starts + lens wraps modulo 2^64 to inside data_bytes
    "ragged_start_wraps": (dict(n=10, data_bytes=1000, starts=_edit(S, 2, (1 << 64) - 50), lens=LN), B.GBIN_E_INVALID_ARG, HOST_ENTRIES),
    "ragged_longer_than_max_read_len": (dict(n=10, data_bytes=1000, starts=S, lens=_edit(LN, 3, 120), max_read_len=100),
                                        B.GBIN_E_INVALID_ARG, HOST_ENTRIES),
}


def long_read_cases():
    """Reads one base longer than gbin_max_read_len(): refused with GBIN_E_TOO_LARGE once their length is known."""
    L1 = int(B.load_library().gbin_max_read_len()) + 1
    return {
        "fixed_longer_than_the_limit": (dict(n=2, data_bytes=2 * L1, stride=L1, read_len=L1), B.GBIN_E_TOO_LARGE, ALL_ENTRIES),
        "ragged_longer_than_the_limit": (dict(n=2, data_bytes=L1 + 100, starts=np.array([0, L1], np.uint64),
                                              lens=np.array([L1, 100], np.uint32)), B.GBIN_E_TOO_LARGE, ALL_ENTRIES),
    }


def descriptors(torch, f):
    """The same descriptor over host buffers and over device buffers -> (host CReads, device CReads, buffers to keep alive)."""
    size = max(f["data_bytes"], 1) + PAD
    data = np.random.default_rng(1).choice(np.frombuffer(b"ACGT", np.uint8), size)
    starts, lens = f.get("starts"), f.get("lens")
    d_data = torch.from_numpy(data).cuda()
    d_starts = None if starts is None else torch.from_numpy(starts.view(np.int64)).cuda()
    d_lens = None if lens is None else torch.from_numpy(lens.view(np.int32)).cuda()

    def rd(dp, sp, lp):
        return B.Binner._reads(None if f.get("null_data") else dp, f["data_bytes"], f["n"], f.get("stride", 0), f.get("read_len", 0),
                               sp, lp, max_read_len=f.get("max_read_len", 0))

    keep = [data, starts, lens, d_data, d_starts, d_lens]
    return rd(data, starts, lens), rd(d_data, d_starts, d_lens), keep


def call(entry, b, m, rd_host, rd_dev, d_rec):
    t, n1, n2 = B.CTable(), C.c_uint64(), C.c_uint64()
    L = b.lib
    if entry == "host":
        return L.gbin_bin_reads_host(b.h, C.byref(rd_host), C.byref(t))
    if entry == "device":
        return L.gbin_bin_reads_device(b.h, C.byref(rd_dev), None, C.byref(t))
    if entry == "host_part":
        return L.gbin_bin_reads_host_part(b.h, C.byref(rd_host), 0, 2, C.byref(t))
    if entry == "device_part":
        return L.gbin_bin_reads_device_part(b.h, C.byref(rd_dev), 0, 2, None, C.byref(t))
    if entry == "count":
        return L.gbin_count_instances_device(b.h, C.byref(rd_dev), None, C.byref(n1))
    if entry == "scan_reads":
        return L.gbin_scan_reads_device(b.h, C.byref(rd_dev), 0, d_rec.data_ptr(), 0, None, C.byref(n1))
    if entry == "scan_skr":
        return L.gbin_scan_skr_device(b.h, C.byref(rd_dev), 0, d_rec.data_ptr(), 0, None, C.byref(n1), C.byref(n2))
    assert entry == "multi"
    return m.bin_raw(rd_host)[0]


def check_valid_batch(b, m):
    """cfg2_small through gbin_bin_reads_host and gbin_multi_bin_reads_host on the contexts that just refused a descriptor."""
    inp = get_input("cfg2_small")
    want = oracle_table("cfg2_small", "default")
    rd, _keep = b._host_reads(inp.data, inp.n, 0, 0, inp.starts, inp.lens, None, 0)
    assert_tables_equal(B.host_table_from_c(b.bin_host_raw(rd)), want, "gbin_bin_reads_host")
    rc, t = m.bin_raw(rd)
    assert rc == B.GBIN_OK, m.lib.gbin_multi_last_error(m.h)
    assert_tables_equal(B.host_table_from_c(t), want, "gbin_multi_bin_reads_host")


@pytest.mark.parametrize("case", list(CASES) + ["fixed_longer_than_the_limit", "ragged_longer_than_the_limit"])
def test_malformed_descriptor_is_refused(case):
    torch = torch_cuda()
    fields, code, entries = {**CASES, **long_read_cases()}[case]
    inp = get_input("cfg2_small")
    b = B.Binner(inp.K, inp.M, inp.cutoff)
    m = Multi(inp.K, inp.M, inp.cutoff)
    try:
        rd_host, rd_dev, _keep = descriptors(torch, fields)
        d_rec = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        got = {e: call(e, b, m, rd_host, rd_dev, d_rec) for e in entries}
        torch.cuda.synchronize()
        assert got == {e: code for e in entries}, got
        check_valid_batch(b, m)
    finally:
        m.close()
        b.close()


# ---------------------------------------------------------------- unusual valid layouts

def offset_shuffled():
    """cfg2_small's reads behind 37 bytes that belong to no read, stored out of read order with an N between reads."""
    inp = get_input("cfg2_small")
    perm = np.random.default_rng(11).permutation(inp.n)
    data = bytearray(b"N" * 37)
    starts = np.zeros(inp.n, np.uint64)
    for i in perm:
        starts[i] = len(data)
        data += inp.data[int(inp.starts[i]): int(inp.starts[i]) + int(inp.lens[i])] + b"N"
    return "cfg2_small", bytes(data), dict(starts=starts, lens=inp.lens)


def wide_stride():
    """deep_31_11's fixed-length reads at a stride of 128 bytes, the gaps filled with N."""
    inp = get_input("deep_31_11")
    stride = 128
    buf = np.full(inp.n * stride, ord("N"), np.uint8)
    src = np.frombuffer(inp.data, np.uint8)
    for i in range(inp.n):
        s = int(inp.starts[i])
        buf[i * stride: i * stride + inp.read_len] = src[s: s + inp.read_len]
    return "deep_31_11", buf[: (inp.n - 1) * stride + inp.read_len].tobytes(), dict(stride=stride, read_len=inp.read_len)


@pytest.mark.parametrize("ids_kind", ["default", "ids"])
@pytest.mark.parametrize("entry", ["host", "host_part", "multi"])
@pytest.mark.parametrize("layout", [offset_shuffled, wide_stride], ids=["offset_shuffled", "wide_stride"])
def test_unusual_valid_layout(layout, entry, ids_kind):
    """ids: caller read_ids together with a non-zero id_base (the ids win)."""
    torch_cuda()
    name, data, kw = layout()
    inp = get_input(name)
    want = oracle_table(name, ids_kind)
    pin = inp.case.get("digest") if (inp.case is not None and ids_kind == "default") else None
    ids = caller_ids(inp.n) if ids_kind == "ids" else None
    b = B.Binner(inp.K, inp.M, inp.cutoff)
    m = None
    try:
        rd, _keep = b._host_reads(data, inp.n, kw.get("stride", 0), kw.get("read_len", 0), kw.get("starts"), kw.get("lens"), ids,
                                  1000 if ids_kind == "ids" else 0)
        if entry == "host_part":
            b.set_tuning("part_chunk_kb", 1)
            tables, digests = [], []
            for p in range(3):
                t = b.bin_host_part_raw(rd, p, 3)
                tables.append(B.host_table_from_c(t))
                digests.append(b.table_digest(t))
            check_parts(inp, 3, tables, digests, want, oracle_tuples(name), pin)
            return
        if entry == "host":
            t = b.bin_host_raw(rd)
        else:
            m = Multi(inp.K, inp.M, inp.cutoff)
            rc, t = m.bin_raw(rd)
            assert rc == B.GBIN_OK, m.lib.gbin_multi_last_error(m.h)
        assert_tables_equal(B.host_table_from_c(t), want, f"{name} via {entry}")
        digest = b.table_digest(t)
        assert digest == O.table_digest(want)
        if pin is not None:
            assert "%016x" % digest == pin
    finally:
        if m is not None:
            m.close()
        b.close()
