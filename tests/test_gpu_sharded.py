"""The multi-GPU sequence of staged entry points, emulated on one GPU: G ranks, each with its own context, scan contiguous read
ranges with arrival_base = first read of the range; the records are partitioned by owner = gbin_owner_of(m-mer, G); every owner
groups what all ranks hold for it, in rank order (the transport dist.py uses without a peer path: partition locally, then an
all-to-all, here a torch.cat on one device).  Every stage is compared with the oracle: the scanned windows, the partition (byte
for byte), every owner's table (the oracle's table restricted to the owner's buckets) and the merged table and digests."""
import functools

import numpy as np
import pytest

import oracle_lib as O
from genome_assembly_b200 import binding as B
from genome_assembly_b200 import dist
from genome_assembly_b200 import synth

pytestmark = pytest.mark.gpu

CASES = {c["name"]: c for c in O.load_pins()}
GPU_CASES = [n for n, c in CASES.items() if c["acgt_only"] and c["k"] >= 2 * c["m"]]
SHARD_CASES = [n for n in GPU_CASES if n != "fuzz_polyA"]  # fuzz_polyA overflows a unit: test_overflow_contract


def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    return torch


# ---------------------------------------------------------------- inputs

class Input:
    """A batch of reads on the host: ragged (starts / lens into `data`) or fixed-stride (`stride`, `read_len`)."""

    def __init__(self, name, data, starts, lens, K, M, cutoff, stride=0, read_len=0, case=None):
        self.name, self.data, self.starts, self.lens = name, data, starts, lens
        self.K, self.M, self.cutoff = K, M, cutoff
        self.stride, self.read_len, self.case = stride, read_len, case
        self.kw = 1 if K <= 32 else 2

    @property
    def n(self):
        return len(self.starts)


def _synthetic(name, rs, K, M, cutoff=1):
    starts = np.arange(rs.n_reads, dtype=np.uint64) * rs.stride
    lens = np.full(rs.n_reads, rs.read_len, dtype=np.uint32)
    return Input(name, rs.as_bytes(), starts, lens, K, M, cutoff, rs.stride, rs.read_len)


def _poly_a(n_reads):
    data = (b"A" * 100 + b"\n") * n_reads
    return Input(f"poly_a_{n_reads}", data, np.arange(n_reads, dtype=np.uint64) * 101, np.full(n_reads, 100, np.uint32), 31, 4, 1,
                 101, 100)


@functools.lru_cache(maxsize=None)
def get_input(name) -> Input:
    if name in CASES:
        c = CASES[name]
        data = O.load_case_bytes(c)
        starts, lens = O.fgets_split(data, c["read_length_define"])
        return Input(name, data, starts, lens, c["k"], c["m"], c["cutoff"], case=c)
    if name == "cfg2_shape":  # 60 000 reads x 100 bp, 4.2 M instances (test_medium_synthetic_cfg2_shape)
        return _synthetic(name, synth.generate(60000, 100, error_rate=0.01, seed=20, starts="triangular"), 31, 11)
    if name.startswith("long_span_m"):  # few, huge buckets: long spans (test_v3_long_spans_are_sorted_span_by_span)
        return _synthetic(name, synth.generate(60000, 100, error_rate=0.01, seed=20, starts="triangular"), 25, int(name[-1]))
    if name.startswith("deep_"):  # ~125x coverage of a 2 000-base genome: d-rounds and spans (test_deep_coverage_rounds_and_spans)
        K, M = (int(x) for x in name[5:].split("_"))
        return _synthetic(name, synth.generate(2500, 100, genome_len=2000, error_rate=0.002, seed=77, starts="uniform"), K, M)
    if name == "poly_a_3000":  # one k-mer with 210 000 instances (test_homopolymer_batch_falls_back_to_the_hbm_pipeline)
        return _poly_a(3000)
    if name == "three_reads":
        return _synthetic(name, synth.generate(3, 100, genome_len=400, error_rate=0.01, seed=3, starts="uniform"), 31, 11)
    raise KeyError(name)


SYNTH_CASES = ["cfg2_shape", "deep_31_11", "deep_31_4", "deep_63_15", "long_span_m4", "long_span_m5"]


def caller_ids(n):
    """Arbitrary caller ids, not sorted (as in test_fixed_stride_form_and_explicit_ids)."""
    return (np.arange(n, dtype=np.int32) * 7 + 100)[::-1].copy()


@functools.lru_cache(maxsize=None)
def oracle_tuples(name):
    inp = get_input(name)
    tup, _ = O.scan_all(inp.data, inp.starts, inp.lens, inp.K, inp.M)
    return tup


@functools.lru_cache(maxsize=None)
def oracle_table(name, ids_kind) -> O.Table:
    """ids_kind: "default" (id = arrival), "base" (1000 + arrival) or "ids" (caller_ids looked up by arrival)."""
    inp = get_input(name)
    if ids_kind == "ids":
        return O.run(inp.data, inp.starts, inp.lens, inp.K, inp.M, inp.cutoff, ids=caller_ids(inp.n))
    t = O.run(inp.data, inp.starts, inp.lens, inp.K, inp.M, inp.cutoff)
    if ids_kind == "base":
        t.read_ids = t.read_ids + 1000
    return t


# ---------------------------------------------------------------- helpers

def assert_tables_equal(got: B.HostTable, want: O.Table, what=""):
    assert (got.K, got.M, got.kw) == (want.K, want.M, want.kw), what
    assert got.n_instances == want.n_instances, what
    assert got.n_distinct == want.n_distinct, what
    np.testing.assert_array_equal(got.mmer_codes, want.mmer_codes, err_msg=what)
    np.testing.assert_array_equal(got.mmer_kmer_off, want.mmer_kmer_off, err_msg=what)
    np.testing.assert_array_equal(got.kmer_codes, want.kmer_codes.reshape(-1), err_msg=what)
    np.testing.assert_array_equal(got.kmer_id_off, want.kmer_id_off, err_msg=what)
    np.testing.assert_array_equal(got.read_ids, want.read_ids, err_msg=what)


def owner_slice(t: O.Table, keep: np.ndarray, n_instances: int, n_distinct: int) -> O.Table:
    """The part of table t in the buckets where keep[bucket] is True (canonical order is kept)."""
    mo = t.mmer_kmer_off.astype(np.int64)
    ko = t.kmer_id_off.astype(np.int64)
    kmer_keep = np.repeat(keep, np.diff(mo))
    id_keep = np.repeat(kmer_keep, np.diff(ko))
    kc = t.kmer_codes.reshape(-1, t.kw)[kmer_keep].reshape(-1)
    mmer_off = np.concatenate([[0], np.cumsum(np.diff(mo)[keep])]).astype(np.uint64)
    id_off = np.concatenate([[0], np.cumsum(np.diff(ko)[kmer_keep])]).astype(np.uint64)
    return O.Table(t.K, t.M, t.cutoff, n_instances, n_distinct, t.mmer_codes[keep], mmer_off, kc, id_off, t.read_ids[id_keep])


def owner_counts(tup, G):
    """(n_instances, n_distinct) of every owner, counted on the oracle's per-window tuples."""
    own = B.owner_of(tup["mmer"], G)
    out = []
    for o in range(G):
        t = tup[own == o]
        out.append((len(t), len(np.unique(t[["mmer", "khi", "klo"]]))))
    return out


def expand_skr(words: np.ndarray, K: int):
    """Super-k-mer records (include/gbin.h layout, u32 words) -> per-window (mmer, arrival, khi, klo) in record order."""
    n_rec, nw = words.shape
    n = (words[:, 2] & 0xFF).astype(np.int64)
    rev = ((words[:, 2] >> 8) & 1).astype(bool)
    shifts = (30 - 2 * np.arange(16)).astype(np.uint32)
    bases = ((words[:, 4:, None] >> shifts) & 3).reshape(n_rec, 16 * (nw - 4)).astype(np.uint8)
    rec = np.repeat(np.arange(n_rec), n)
    t = np.arange(len(rec)) - np.repeat(np.cumsum(n) - n, n)
    comp = np.repeat(rev, n).astype(np.uint64) * np.uint64(3)
    flat = bases.reshape(-1)
    pos = rec * bases.shape[1] + t
    khi = np.zeros(len(rec), np.uint64)
    klo = np.zeros(len(rec), np.uint64)
    for u in range(K):
        b = flat[pos + u].astype(np.uint64) ^ comp
        if u < K - 32:
            khi = (khi << np.uint64(2)) | b
        else:
            klo = (klo << np.uint64(2)) | b
    return words[rec, 1], words[rec, 0], khi, klo


def record_fields(words: np.ndarray, kw: int):
    """Instance records (u32 words: kmer u64 words, mmer, arrival) -> (mmer, arrival, khi, klo)."""
    k = words[:, : 2 * kw].copy().view(np.uint64)
    khi = k[:, 0] if kw == 2 else np.zeros(len(words), np.uint64)
    return words[:, 2 * kw], words[:, 2 * kw + 1], khi, k[:, -1]


def assert_windows_equal(got, want, what):
    mmer, arrival, khi, klo = got
    assert len(mmer) == len(want), what
    np.testing.assert_array_equal(mmer, want["mmer"], err_msg=what)
    np.testing.assert_array_equal(arrival, want["arrival"], err_msg=what)
    np.testing.assert_array_equal(klo, want["klo"], err_msg=what)
    np.testing.assert_array_equal(khi, want["khi"], err_msg=what)


class DeviceBatch:
    """The batch's reads on the device; shard(lo, hi) is the CReads of reads [lo, hi) (fixed-stride or ragged form)."""

    def __init__(self, torch, inp: Input):
        self.inp = inp
        self.d = torch.from_numpy(np.frombuffer(inp.data, dtype=np.uint8).copy()).cuda()
        self.s = torch.from_numpy(inp.starts.astype(np.int64)).cuda()
        self.l = torch.from_numpy(inp.lens.astype(np.int32)).cuda()

    def shard(self, lo, hi):
        inp = self.inp
        if inp.stride:
            return B.Binner._reads(self.d.data_ptr() + lo * inp.stride, max(self.d.numel() - lo * inp.stride, 0), hi - lo,
                                   stride=inp.stride, read_len=inp.read_len)
        return B.Binner._reads(self.d, self.d.numel(), hi - lo, starts=self.s[lo:hi], lens=self.l[lo:hi])


def rows(torch, buf, n, rb):
    return buf[: n * rb].cpu().numpy().reshape(n, rb)


# ---------------------------------------------------------------- the sharded run

def scan_and_partition(torch, inp, binners, G, form, arrival_check=True):
    """Every rank scans its shard (arrival_base = lo) and partitions its records by owner.  Checks the windows against the oracle and
    the partition byte for byte.  -> (per rank: (scan buffer, partition buffer, counts)), record bytes."""
    stream = B.stream_handle(torch.cuda.current_stream())
    tup = oracle_tuples(inp.name)
    batch = DeviceBatch(torch, inp)
    n = inp.n
    ranks = []
    rb = binners[0].skr_record_bytes if form == "skr" else binners[0].record_bytes
    for g in range(G):
        b = binners[g]
        lo, hi = g * n // G, (g + 1) * n // G
        rd = batch.shard(lo, hi)
        n_inst = b.count_instances_device(rd, stream)
        buf = torch.empty(max(n_inst, 1) * rb, dtype=torch.uint8, device="cuda")
        if form == "skr":
            n_rec, got_inst = b.scan_skr_device(rd, lo, buf, max(n_inst, 1), stream)
            assert got_inst == n_inst
        else:
            n_rec = b.scan_device(rd, lo, buf, n_inst, stream)
            assert n_rec == n_inst
        r_in = rows(torch, buf, n_rec, rb)
        words = r_in.view(np.uint32)
        if arrival_check:
            want = tup[(tup["arrival"] >= lo) & (tup["arrival"] < hi)]  # scan_all(reads lo..hi-1) with arrival + lo
            got = expand_skr(words, inp.K) if form == "skr" else record_fields(words, inp.kw)
            assert_windows_equal(got, want, f"rank {g} of {G}: windows of reads [{lo}, {hi})")
        out = torch.empty_like(buf)
        if form == "skr":
            counts = b.partition_skr_device(buf, n_rec, G, out, stream)
            mmer = words[:, 1]
        else:
            counts = b.partition_device(buf, n_rec, G, out, stream)
            mmer = words[:, 2 * inp.kw]
        own = B.owner_of(mmer, G)
        assert counts == np.bincount(own, minlength=G).tolist(), (g, counts)
        np.testing.assert_array_equal(rows(torch, out, n_rec, rb), r_in[np.argsort(own, kind="stable")],
                                      err_msg=f"rank {g}: partition is not the stable owner order of the records")
        ranks.append((buf, out, counts))
    return ranks, rb


def owner_input(torch, ranks, rb, o):
    """Part o of every rank, in rank order (what the all-to-all hands to owner o)."""
    parts = []
    for _, out, counts in ranks:
        off = sum(counts[:o])
        parts.append(out[off * rb: (off + counts[o]) * rb])
    recv = torch.cat(parts) if parts else torch.empty(0, dtype=torch.uint8, device="cuda")
    n = sum(c[o] for _, _, c in ranks)
    if recv.numel() == 0:
        recv = torch.empty(rb, dtype=torch.uint8, device="cuda")
    return recv, n


def check_owner_tables(inp, G, tables, ids_kind, digests=None):
    """Every owner's table == the oracle's table restricted to its buckets; together the oracle's table (and the pins)."""
    want = oracle_table(inp.name, ids_kind)
    own_b = B.owner_of(want.mmer_codes, G)
    cnt = owner_counts(oracle_tuples(inp.name), G)
    for o, t in enumerate(tables):
        assert_tables_equal(t, owner_slice(want, own_b == o, *cnt[o]), f"owner {o} of {G}")
    merged = dist.merge_owner_tables(tables)
    assert_tables_equal(merged, want, f"merged tables of {G} owners")
    if inp.case is not None and ids_kind == "default":
        assert O.Table(merged.K, merged.M, merged.cutoff, merged.n_instances, merged.n_distinct, merged.mmer_codes, merged.mmer_kmer_off,
                       merged.kmer_codes, merged.kmer_id_off, merged.read_ids).md5() == inp.case["md5"]
        if digests is not None and "digest" in inp.case:
            assert "%016x" % (sum(digests) % (1 << 64)) == inp.case["digest"]


def group_ids(torch, inp, ids_kind):
    """(d_ids_by_arrival, id_base) of a grouping call; the caller-id array is global: every owner is given all of it."""
    if ids_kind == "ids":
        return torch.from_numpy(caller_ids(inp.n)).cuda(), 0
    return None, (1000 if ids_kind == "base" else 0)


def run_sharded(name, G, *, ids_kind="default", pipeline=3, tuning=(), form="skr"):
    """The whole emulated multi-GPU run; -> (per-owner host tables, per-owner run_stats, per-owner pipeline_info)."""
    torch = torch_cuda()
    inp = get_input(name)
    stream = B.stream_handle(torch.cuda.current_stream())
    binners = [B.Binner(inp.K, inp.M, inp.cutoff, pipeline=pipeline) for _ in range(G)]
    try:
        for b in binners:
            for k, v in tuning:
                b.set_tuning(k, v)
        ranks, rb = scan_and_partition(torch, inp, binners, G, form)
        d_ids, id_base = group_ids(torch, inp, ids_kind)
        tables, digests, stats, infos = [], [], [], []
        for o in range(G):
            b = binners[o]
            recv, n = owner_input(torch, ranks, rb, o)
            if form == "skr":
                dev = b.group_skr_device(recv, n, d_ids, id_base, stream)
            else:
                dev = b.group_device(recv, n, d_ids, id_base, stream)
            digests.append(b.table_digest(dev, stream))
            tables.append(b.table_to_host(dev))
            stats.append(b.run_stats())
            infos.append(b.pipeline_info())
        check_owner_tables(inp, G, tables, ids_kind, digests)
        return tables, stats, infos
    finally:
        for b in binners:
            b.close()


# ---------------------------------------------------------------- tests

@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("name", SHARD_CASES + SYNTH_CASES)
def test_super_kmer_shards_match_oracle(name, G):
    """scan_skr_device(arrival_base = lo) -> partition_skr_device -> group_skr_device per owner, pipeline 3."""
    _, stats, infos = run_sharded(name, G)
    if name.startswith("long_span"):  # which path a span takes is not pinned: an owner that kept pipeline 3 sorted long spans
        print(name, G, [i["last_used"] for i in infos], stats)
        v3 = [s["n_lsd_kmers"] for s, i in zip(stats, infos) if i["last_used"] == 3]
        assert not v3 or sum(v3) > 0, stats


@pytest.mark.parametrize("pipeline", [3, 2])
@pytest.mark.parametrize("ids_kind", ["base", "ids"])
@pytest.mark.parametrize("name", ["cfg2_small", "cfg4_small", "fuzz_ragged_k25", "cfg2_shape", "deep_31_11", "deep_31_4", "deep_63_15",
                                  "long_span_m5"])
def test_caller_ids_reach_every_owner(name, ids_kind, pipeline):
    """id_base = 1000, and a global, unsorted ids_by_arrival array handed whole to every owner (G = 3)."""
    run_sharded(name, 3, ids_kind=ids_kind, pipeline=pipeline)


@pytest.mark.parametrize("name", ["cfg2_small", "cfg5_small", "deep_31_11", "deep_63_15", "cfg2_shape"])
def test_owner_settings_pipeline2_and_two_key_words(name):
    """Owners on pipeline 2, and pipeline 3 with its two-word key layout (v3_nc = 2)."""
    _, _, infos = run_sharded(name, 3, pipeline=2)
    if not name.startswith("deep"):
        assert all(i["last_used"] == 2 for i in infos), infos
    run_sharded(name, 3, tuning=(("v3_nc", 2), ("v3_h", 2)))


def test_owner_passes():
    """A pass limit of 300 000 instances on the cfg2 shape at G = 2: every owner groups its ~2.1 M instances in several passes
    (passes are cut at 65 536-entry tile boundaries, so the limit has no effect on the small fixtures)."""
    _, stats, infos = run_sharded("cfg2_shape", 2, tuning=(("v3_pass_max", 300_000),))
    assert all(i["last_used"] == 3 for i in infos), infos
    assert all(s["n_passes"] >= 2 for s in stats), stats


@pytest.mark.parametrize("ids_kind", ["default", "ids"])
@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("name", ["cfg2_small", "cfg4_small", "fuzz_ragged_k15", "fuzz_polyA", "deep_63_15", "cfg2_shape"])
def test_instance_record_shards_match_oracle(name, G, ids_kind):
    """dist.py's "records" form, which is also the fallback: scan_device(arrival_base = lo) -> partition_device -> group_device."""
    run_sharded(name, G, ids_kind=ids_kind, form="records")


@pytest.mark.parametrize("form", ["skr", "records"])
def test_owners_without_records(form):
    """kat_twice (20 instances) at G = 8: most owners receive no record and return an empty table with digest 0."""
    tables, _, _ = run_sharded("kat_twice", 8, form=form)
    want = oracle_table("kat_twice", "default")
    empty = [t for t in tables if t.n_instances == 0]
    assert len(empty) >= 4 and len(want.mmer_codes) > 0
    for t in empty:
        assert (t.n_buckets, t.n_kmers, t.n_ids, t.n_distinct) == (0, 0, 0, 0)
        np.testing.assert_array_equal(t.kmer_id_off, [0])


@pytest.mark.parametrize("form", ["skr", "records"])
def test_shards_without_reads(form):
    """3 reads at G = 8: five shards hold no read (the scan returns 0 records) and most owners get 0 records to group."""
    torch = torch_cuda()
    inp = get_input("three_reads")
    stream = B.stream_handle(torch.cuda.current_stream())
    binners = [B.Binner(inp.K, inp.M, inp.cutoff) for _ in range(8)]
    try:
        ranks, rb = scan_and_partition(torch, inp, binners, 8, form)
        assert sum(1 for _, _, c in ranks if sum(c) == 0) == 5
        tables, digests = [], []
        for o in range(8):
            recv, n = owner_input(torch, ranks, rb, o)
            dev = (binners[o].group_skr_device(recv, n, None, 0, stream) if form == "skr" else
                   binners[o].group_device(recv, n, None, 0, stream))
            digests.append(binners[o].table_digest(dev, stream))
            tables.append(binners[o].table_to_host(dev))
            if n == 0:
                assert digests[-1] == 0 and tables[-1].n_instances == 0
                np.testing.assert_array_equal(tables[-1].kmer_id_off, [0])
        check_owner_tables(inp, 8, tables, "default")
        assert sum(digests) % (1 << 64) == O.table_digest(oracle_table("three_reads", "default"))
    finally:
        for b in binners:
            b.close()


@pytest.mark.parametrize("name", ["fuzz_polyA", "poly_a_3000"])
def test_overflow_contract(name):
    """A k-mer with more instances than a shared-memory unit holds: group_skr_device raises GBIN_E_STATE on the owner of its bucket,
    and the batch redone in instance-record form gives the oracle's table."""
    torch = torch_cuda()
    inp = get_input(name)
    G = 2
    stream = B.stream_handle(torch.cuda.current_stream())
    tup = oracle_tuples(name)
    _, first, cnt = np.unique(tup[["mmer", "khi", "klo"]], return_index=True, return_counts=True)
    heavy = int(B.owner_of(tup["mmer"][first[np.argmax(cnt)]], G))
    binners = [B.Binner(inp.K, inp.M, inp.cutoff) for _ in range(G)]
    try:
        ranks, rb = scan_and_partition(torch, inp, binners, G, "skr")
        for o in range(G):
            recv, n = owner_input(torch, ranks, rb, o)
            if o == heavy:
                with pytest.raises(B.GbinError) as e:
                    binners[o].group_skr_device(recv, n, None, 0, stream)
                assert e.value.code == B.GBIN_E_STATE
            else:
                try:
                    binners[o].group_skr_device(recv, n, None, 0, stream)
                except B.GbinError as e:
                    assert e.code == B.GBIN_E_STATE
    finally:
        for b in binners:
            b.close()
    run_sharded(name, G, form="records")


def test_donated_scratch_is_used_for_one_call():
    """Each rank's scan buffer, dead after the partition, is lent to an owner's grouping call; then the buffer is overwritten with
    0xFF and the owner groups again without a loan (the loan ended with the call).  A loan that is too small or not 16-byte aligned
    is ignored.  Every table must be the oracle's."""
    torch = torch_cuda()
    inp = get_input("cfg2_shape")
    G = 2
    stream = B.stream_handle(torch.cuda.current_stream())
    want = oracle_table(inp.name, "default")
    own_b = B.owner_of(want.mmer_codes, G)
    cnt = owner_counts(oracle_tuples(inp.name), G)
    binners = [B.Binner(inp.K, inp.M, inp.cutoff) for _ in range(G)]
    try:
        ranks, rb = scan_and_partition(torch, inp, binners, G, "skr", arrival_check=False)
        for o in range(G):
            b = binners[o]
            recv, n = owner_input(torch, ranks, rb, o)
            keep = recv.clone()  # the grouping call clobbers its input
            slice_o = owner_slice(want, own_b == o, *cnt[o])
            lent = ranks[(o + 1) % G][0]
            b.donate_scratch(lent, lent.numel())
            assert_tables_equal(b.table_to_host(b.group_skr_device(recv, n, None, 0, stream)), slice_o, f"owner {o}, donated")
            lent.fill_(0xFF)
            recv.copy_(keep)
            assert_tables_equal(b.table_to_host(b.group_skr_device(recv, n, None, 0, stream)), slice_o, f"owner {o}, after the loan")
            for ptr, nbytes in ((lent.data_ptr(), 4096), (lent.data_ptr() + 8, lent.numel() - 8)):  # too small; misaligned
                b.donate_scratch(ptr, nbytes)
                recv.copy_(keep)
                assert_tables_equal(b.table_to_host(b.group_skr_device(recv, n, None, 0, stream)), slice_o, f"owner {o}, bad loan")
                lent.fill_(0xFF)
    finally:
        for b in binners:
            b.close()


@pytest.mark.parametrize("L", [100, 300])
def test_scan_capacity_is_respected(L):
    """scan_skr_device with a capacity one record short of the need raises GBIN_E_INVALID_ARG and writes nothing past capacity; with the
    exact need the records equal those of a generous capacity.  100-bp reads run the lane-per-position scan kernel, 300-bp reads
    (more than 256 m-mer positions) the hop-chain kernel."""
    torch = torch_cuda()
    rs = synth.generate(2000, L, error_rate=0.01, seed=L, starts="uniform")
    inp = _synthetic(f"cap_{L}", rs, 31, 11)
    base = 123_457
    stream = B.stream_handle(torch.cuda.current_stream())
    b = B.Binner(31, 11, 1)
    try:
        batch = DeviceBatch(torch, inp)
        rd = batch.shard(0, inp.n)
        rb = b.skr_record_bytes
        n_inst = b.count_instances_device(rd, stream)
        big = torch.zeros(n_inst * rb, dtype=torch.uint8, device="cuda")
        need, got_inst = b.scan_skr_device(rd, base, big, n_inst, stream)
        assert got_inst == n_inst and 0 < need < n_inst
        ref = rows(torch, big, need, rb)
        tup, _ = O.scan_all(inp.data, inp.starts, inp.lens, 31, 11)
        tup["arrival"] += base
        assert_windows_equal(expand_skr(ref.view(np.uint32), 31), tup, f"{L}-bp reads, arrival_base {base}")
        buf = torch.full(((need + 64) * rb,), 0xA5, dtype=torch.uint8, device="cuda")
        with pytest.raises(B.GbinError) as e:
            b.scan_skr_device(rd, base, buf, need - 1, stream)
        assert e.value.code == B.GBIN_E_INVALID_ARG
        tail = buf[(need - 1) * rb:].cpu().numpy()
        assert (tail == 0xA5).all(), f"{int((tail != 0xA5).sum())} bytes written past the capacity"
        buf.fill_(0xA5)
        assert b.scan_skr_device(rd, base, buf, need, stream) == (need, n_inst)
        np.testing.assert_array_equal(rows(torch, buf, need, rb), ref)
        assert (buf[need * rb:].cpu().numpy() == 0xA5).all()
    finally:
        b.close()
