"""The table in owner parts, one part per call (gbin_bin_reads_host_part / gbin_bin_reads_device_part): part p of P must be the
oracle's table restricted to the m-mer buckets with gbin_owner_of(m-mer, P) == p, with n_instances / n_distinct counted on the
oracle's windows of those buckets, and the parts' digests must add up to the whole table's digest (the fixtures' pins)."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from genome_assembly_b200 import binding as B
from genome_assembly_b200 import synth
from test_gpu_sharded import (SHARD_CASES, SYNTH_CASES, Input, _synthetic, assert_tables_equal, caller_ids, get_input, oracle_table,
                              oracle_tuples, owner_counts, owner_slice, torch_cuda)

pytestmark = pytest.mark.gpu

MASK64 = (1 << 64) - 1


def forms(names):
    """Fixture files are ragged; the synthetic read sets are fixed-stride and are run in both forms."""
    return [(n, f) for n in names for f in (("ragged", "fixed") if get_input_kind(n) == "synthetic" else ("ragged",))]


def get_input_kind(name):
    return "synthetic" if name in SYNTH_CASES or name in ("three_reads", "poly_a_3000") else "fixture"


def host_kwargs(inp, form, ids_kind):
    kw = dict(read_ids=caller_ids(inp.n) if ids_kind == "ids" else None, id_base=1000 if ids_kind == "base" else 0)
    if form == "fixed":
        kw.update(stride=inp.stride, read_len=inp.read_len)
    else:
        kw.update(starts=inp.starts, lens=inp.lens)
    return kw


def run_host_parts(inp, P, *, form="ragged", ids_kind="default", pipeline=3, tuning=(), order=None):
    """Every part of P through gbin_bin_reads_host_part on one context -> (tables, digests, pipeline infos, run stats), by part."""
    torch_cuda()
    b = B.Binner(inp.K, inp.M, inp.cutoff, pipeline=pipeline)
    try:
        for k, v in tuning:
            b.set_tuning(k, v)
        kw = host_kwargs(inp, form, ids_kind)
        rd, _keep = b._host_reads(inp.data, inp.n, kw.get("stride", 0), kw.get("read_len", 0), kw.get("starts"), kw.get("lens"),
                                  kw["read_ids"], kw["id_base"])
        out = {}
        for p in (order if order is not None else range(P)):
            t = b.bin_host_part_raw(rd, p, P)
            out[p] = (B.host_table_from_c(t), b.table_digest(t), b.pipeline_info(), b.run_stats())
        return [list(x) for x in zip(*(out[p] for p in range(P)))]
    finally:
        b.close()


def check_parts(inp, P, tables, digests, want, tup, pinned_digest=None):
    """Every part == the oracle's table on its buckets; the digests add up to the whole table's."""
    own = B.owner_of(want.mmer_codes, P)
    cnt = owner_counts(tup, P)
    for p, t in enumerate(tables):
        assert_tables_equal(t, owner_slice(want, own == p, *cnt[p]), f"{inp.name}: part {p} of {P}")
    total = sum(digests) & MASK64
    assert total == O.table_digest(want), f"{inp.name}: digests of {P} parts"
    if pinned_digest is not None:
        assert "%016x" % total == pinned_digest


def check_named(name, P, tables, digests, ids_kind="default"):
    inp = get_input(name)
    pin = inp.case.get("digest") if (inp.case is not None and ids_kind == "default") else None
    check_parts(inp, P, tables, digests, oracle_table(name, ids_kind), oracle_tuples(name), pin)


# ---------------------------------------------------------------- 1. parts against the oracle

@pytest.mark.parametrize("P", [1, 2, 3, 8])
@pytest.mark.parametrize("name,form", forms(SHARD_CASES + SYNTH_CASES))
def test_parts_match_oracle(name, form, P):
    inp = get_input(name)
    tables, digests, _, _ = run_host_parts(inp, P, form=form)
    check_named(name, P, tables, digests)
    if P == 1:  # one part is the whole table, byte for byte what gbin_bin_reads_host returns
        b = B.Binner(inp.K, inp.M, inp.cutoff)
        kw = host_kwargs(inp, form, "default")
        whole = b.bin_host(inp.data, inp.n, **kw)
        b.close()
        for f in ("n_instances", "n_distinct", "mmer_codes", "mmer_kmer_off", "kmer_codes", "kmer_id_off", "read_ids"):
            np.testing.assert_array_equal(getattr(tables[0], f), getattr(whole, f), err_msg=f)


# ---------------------------------------------------------------- 2. chunk boundaries

@pytest.mark.parametrize("ids_kind", ["default", "ids", "base"])
@pytest.mark.parametrize("name,form,P", [("short_reads", "ragged", 3), ("cfg1_reads", "ragged", 2), ("fuzz_ragged_k15", "ragged", 3),
                                         ("kat_twice", "ragged", 8), ("deep_31_11", "fixed", 3), ("deep_63_15", "ragged", 2)])
def test_one_kib_chunks(name, form, P, ids_kind):
    """part_chunk_kb = 1: a handful of reads per chunk, so chunks start and end everywhere, also next to reads shorter than K
    (short_reads); kat_twice at P = 8 has chunks that hold no record of a part."""
    tables, digests, _, _ = run_host_parts(get_input(name), P, form=form, ids_kind=ids_kind, tuning=(("part_chunk_kb", 1),))
    check_named(name, P, tables, digests, ids_kind)


def test_reads_laid_out_out_of_order():
    """Ragged reads whose bytes are not in read order: a chunk is cut where the span of its reads would exceed the budget."""
    inp = get_input("cfg2_small")
    perm = np.random.default_rng(5).permutation(inp.n)
    data = bytearray()
    starts = np.zeros(inp.n, np.uint64)
    for i in perm:  # read i's bytes are stored in the order of perm
        starts[i] = len(data)
        data += inp.data[int(inp.starts[i]): int(inp.starts[i]) + int(inp.lens[i])] + b"\n"
    shuffled = Input("cfg2_small_shuffled", bytes(data), starts, inp.lens, inp.K, inp.M, inp.cutoff)
    tables, digests, _, _ = run_host_parts(shuffled, 3, tuning=(("part_chunk_kb", 4),))
    check_parts(shuffled, 3, tables, digests, oracle_table("cfg2_small", "default"), oracle_tuples("cfg2_small"), inp.case["digest"])


# ---------------------------------------------------------------- 3. device form

@pytest.mark.parametrize("P", [1, 3])
@pytest.mark.parametrize("name", ["cfg2_small", "cfg5_small", "fuzz_ragged_k25", "deep_63_15", "cfg2_shape"])
def test_device_form(name, P):
    """Fixtures: the file image split on the device (gbin_split_reads_device); synthetic sets: a fixed-stride device tensor.  On a
    caller stream, with 8 KiB chunks."""
    torch = torch_cuda()
    inp = get_input(name)
    s = torch.cuda.Stream()
    stream = B.stream_handle(s)
    b = B.Binner(inp.K, inp.M, inp.cutoff)
    try:
        b.set_tuning("part_chunk_kb", 8)
        with torch.cuda.stream(s):
            d = torch.from_numpy(np.frombuffer(inp.data, dtype=np.uint8).copy()).cuda()
        if inp.case is not None:
            rd = b.split_reads_device(d, d.numel(), inp.case["read_length_define"], stream)
            assert rd.n_reads == inp.n
        else:
            rd = B.Binner._reads(d, d.numel(), inp.n, stride=inp.stride, read_len=inp.read_len)
        tables, digests = [], []
        for p in range(P):
            dev = b.bin_device_part_raw(rd, p, P, stream)
            assert dev.on_device == 1 and dev.ctx_owned == 1
            digests.append(b.table_digest(dev, stream))
            tables.append(b.table_to_host(dev))
        check_named(name, P, tables, digests)
    finally:
        b.close()


# ---------------------------------------------------------------- 4. pipelines

@pytest.mark.parametrize("pipeline", [2, 1])
@pytest.mark.parametrize("name,form", [("cfg2_small", "ragged"), ("cfg4_small", "ragged"), ("fuzz_ragged_k15", "ragged"),
                                       ("deep_31_11", "fixed"), ("cfg2_shape", "ragged")])
def test_pipelines_2_and_1(name, form, pipeline):
    tables, digests, infos, _ = run_host_parts(get_input(name), 3, form=form, pipeline=pipeline)
    check_named(name, 3, tables, digests)
    if pipeline == 1:
        assert all(i["last_used"] == 1 for i in infos), infos


# ---------------------------------------------------------------- 5. overflow and long reads

@pytest.mark.parametrize("P", [2, 3])
@pytest.mark.parametrize("name", ["fuzz_polyA", "poly_a_3000"])
def test_overflow_only_the_heavy_part_falls_back(name, P):
    """A k-mer with more instances than a shared-memory unit holds: the part of its bucket goes through pipeline 1, the others
    stay on pipeline 3."""
    inp = get_input(name)
    tup = oracle_tuples(name)
    _, first, cnt = np.unique(tup[["mmer", "khi", "klo"]], return_index=True, return_counts=True)
    heavy = int(B.owner_of(tup["mmer"][first[np.argmax(cnt)]], P))
    tables, digests, infos, _ = run_host_parts(inp, P, form="fixed" if inp.stride else "ragged")
    check_named(name, P, tables, digests)
    assert infos[heavy]["last_used"] == 1, infos
    for p, i in enumerate(infos):
        if p != heavy and tables[p].n_instances:
            assert i["last_used"] == 3, (p, infos)


@pytest.mark.parametrize("K,M", [(31, 11), (63, 15)])
@pytest.mark.parametrize("form", ["fixed", "ragged"])
def test_long_reads(form, K, M):
    """4 000-base reads, 64 KiB chunks: the super-k-mer scan runs with fewer warps per block or leaves the reads to the instance-record
    scan (test_long_reads_pick_a_scan_kernel_that_fits); either way every part is the oracle's."""
    torch_cuda()
    rs = synth.generate(300, 4000, genome_len=12000, error_rate=0.01, seed=4000, starts="uniform")
    inp = _synthetic(f"long_4000_k{K}", rs, K, M)
    tup, _ = O.scan_all(inp.data, inp.starts, inp.lens, K, M)
    want = O.run(inp.data, inp.starts, inp.lens, K, M, 1)
    tables, digests, infos, _ = run_host_parts(inp, 2, form=form, tuning=(("part_chunk_kb", 64),))
    check_parts(inp, 2, tables, digests, want, tup)
    assert all(i["last_used"] in (1, 3) for i in infos), infos


# ---------------------------------------------------------------- 6. passes inside a part

def test_passes_inside_a_part():
    tables, digests, infos, stats = run_host_parts(get_input("cfg2_shape"), 2, form="fixed", tuning=(("v3_pass_max", 300_000),))
    check_named("cfg2_shape", 2, tables, digests)
    assert all(i["last_used"] == 3 for i in infos), infos
    assert all(s["n_passes"] >= 2 for s in stats), stats


# ---------------------------------------------------------------- 7. degenerate inputs and arguments

def test_no_reads():
    torch = torch_cuda()
    b = B.Binner(31, 11, 1)
    try:
        data = np.zeros(1, np.uint8)
        for p in range(3):
            t = b.bin_host_part(data, 0, p, 3, starts=np.zeros(0, np.uint64), lens=np.zeros(0, np.uint32))
            assert (t.n_instances, t.n_distinct, t.n_buckets, t.n_kmers, t.n_ids) == (0, 0, 0, 0, 0)
            np.testing.assert_array_equal(t.kmer_id_off, [0])
            np.testing.assert_array_equal(t.mmer_kmer_off, [0])
        d = torch.zeros(16, dtype=torch.uint8, device="cuda")
        dev = b.bin_device_part_raw(B.Binner._reads(d, 16, 0, stride=100, read_len=100), 0, 2)
        assert b.table_digest(dev) == 0 and b.table_to_host(dev).n_kmers == 0
    finally:
        b.close()


def test_many_more_parts_than_buckets():
    inp = get_input("three_reads")
    tables, digests, _, _ = run_host_parts(inp, 64, form="fixed")
    check_named("three_reads", 64, tables, digests)
    empty = [t for t in tables if t.n_instances == 0]
    assert len(empty) > 32
    for t in empty:
        np.testing.assert_array_equal(t.mmer_kmer_off, [0])
        np.testing.assert_array_equal(t.kmer_id_off, [0])


def test_bad_arguments():
    torch_cuda()
    inp = get_input("cfg2_small")
    b = B.Binner(inp.K, inp.M, inp.cutoff)
    L = b.lib
    try:
        rd, _keep = b._host_reads(inp.data, inp.n, 0, 0, inp.starts, inp.lens, None, 0)
        t = B.CTable()
        for part, n_parts in ((3, 3), (0, 0), (0, 65537), (70000, 65536)):
            assert L.gbin_bin_reads_host_part(b.h, C.byref(rd), part, n_parts, C.byref(t)) == B.GBIN_E_INVALID_ARG, (part, n_parts)
            assert L.gbin_bin_reads_device_part(b.h, C.byref(rd), part, n_parts, None, C.byref(t)) == B.GBIN_E_INVALID_ARG
        assert L.gbin_bin_reads_host_part(None, C.byref(rd), 0, 2, C.byref(t)) == B.GBIN_E_INVALID_ARG
        assert L.gbin_bin_reads_host_part(b.h, None, 0, 2, C.byref(t)) == B.GBIN_E_INVALID_ARG
        assert L.gbin_bin_reads_host_part(b.h, C.byref(rd), 0, 2, None) == B.GBIN_E_INVALID_ARG
        assert L.gbin_bin_reads_device_part(b.h, None, 0, 2, None, C.byref(t)) == B.GBIN_E_INVALID_ARG
        big = B.Binner._reads(_keep[0], len(inp.data), 1 << 32, starts=_keep[1], lens=_keep[2])
        assert L.gbin_bin_reads_host_part(b.h, C.byref(big), 0, 2, C.byref(t)) == B.GBIN_E_TOO_LARGE
        bad = b"ACGTNACGT" * 20
        with pytest.raises(B.GbinError) as e:
            b.bin_host_part(bad, 1, 0, 1, starts=np.zeros(1, np.uint64), lens=np.array([len(bad)], np.uint32))
        assert e.value.code == B.GBIN_E_NON_ACGT
    finally:
        b.close()


def test_parts_in_reverse_order_then_a_whole_batch():
    """Parts asked for in reverse order give the same tables; a gbin_bin_reads_host call on the same context afterwards still
    matches its pin."""
    inp = get_input("cfg2_small")
    tables, digests, _, _ = run_host_parts(inp, 3, order=[2, 1, 0])
    check_named("cfg2_small", 3, tables, digests)
    b = B.Binner(inp.K, inp.M, inp.cutoff)
    try:
        for p in range(3):
            b.bin_host_part(inp.data, inp.n, p, 3, starts=inp.starts, lens=inp.lens)
        got = b.bin_host(inp.data, inp.n, starts=inp.starts, lens=inp.lens)
        t = O.Table(got.K, got.M, got.cutoff, got.n_instances, got.n_distinct, got.mmer_codes, got.mmer_kmer_off, got.kmer_codes,
                    got.kmer_id_off, got.read_ids)
        assert t.md5() == inp.case["md5"]
    finally:
        b.close()


# ---------------------------------------------------------------- 8. gbin_plan_parts

def test_plan_parts():
    torch_cuda()
    b = B.Binner(31, 11, 1)
    try:
        for name in ("cfg2_small", "cfg5_small", "cfg2_shape"):
            assert b.plan_parts(len(oracle_tuples(name))) == 1
        ps = [b.plan_parts(n) for n in (0, 10**6, 10**9, 10**10, 4 * 10**10, 10**11)]
        assert ps == sorted(ps) and ps[0] == 1 and ps[-1] > 1, ps
        assert b.lib.gbin_plan_parts(b.h, 1000, None) == B.GBIN_E_INVALID_ARG
        assert b.lib.gbin_plan_parts(None, 1000, C.byref(C.c_uint32())) == B.GBIN_E_INVALID_ARG
    finally:
        b.close()


# ---------------------------------------------------------------- 9. full config 2 in three parts

def test_full_cfg2_in_three_parts(tmp_path):
    """BASELINE config 2 (1 M reads x 100 bp) in P = 3 parts: the sorted concatenation of the parts' dumps is the pinned dump."""
    torch_cuda()
    with open(os.path.join(O.GOLDEN, "fullsize_pins.json")) as f:
        case = {c["name"]: c for c in json.load(f)["cases"]}["full_cfg2"]
    rs = synth.generate(case["n_reads"], case["read_len"], error_rate=case["error_rate"], seed=case["seed"], starts=case["starts"])
    b = B.Binner(case["k"], case["m"], case["cutoff"])
    kmers, dumps = 0, []
    try:
        rd = B.Binner._reads(rs.buf, rs.buf.size, rs.n_reads, stride=rs.stride, read_len=rs.read_len)
        for p in range(3):
            t = b.bin_host_part_raw(rd, p, 3)
            assert b.pipeline_info()["last_used"] == 3
            kmers += t.n_kmers
            dumps.append(str(tmp_path / f"part{p}.dump"))
            assert b.lib.gbin_table_dump(C.byref(t), dumps[-1].encode()) == 0
    finally:
        b.close()
    assert kmers == case["surviving_kmers"]
    srt = subprocess.run(["sort", "-S", "2G", *dumps], capture_output=True, check=True, env=dict(os.environ, LC_ALL="C"))
    assert hashlib.md5(srt.stdout).hexdigest() == case["md5"]
