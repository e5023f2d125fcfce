"""CPU: bench.py --dump-outputs writes the table as float64 arrays that hold every code, offset and id exactly, and samples long
arrays at fixed rows (the oracle's table stands in for the device table)."""
import numpy as np
import pytest

import bench
import oracle_lib as O
from genome_assembly_b200.binding import HostTable


class _TableSource:
    def __init__(self, t):
        self.t = t

    def table_to_host(self, _):
        t = self.t
        return HostTable(t.K, t.M, t.cutoff, t.kw, t.n_instances, t.n_distinct, t.mmer_codes, t.mmer_kmer_off, t.kmer_codes,
                         t.kmer_id_off, t.read_ids)


@pytest.mark.parametrize("name,cutoff", [("cfg2_small", None), ("cfg4_small", None), ("kat_twice", None), ("kat_twice", 1000)])
def test_dump_outputs_is_exact_and_sampled_at_fixed_rows(name, cutoff, tmp_path, monkeypatch):
    """cutoff 1000: no k-mer survives, and the dump still writes every array (empty)."""
    case = next(c for c in O.load_pins() if c["name"] == name)
    data = O.load_case_bytes(case)
    starts, lens = O.fgets_split(data, case["read_length_define"])
    t = O.run(data, starts, lens, case["k"], case["m"], cutoff or case["cutoff"])
    assert (t.n_kmers == 0) == (cutoff == 1000)
    monkeypatch.setattr(bench, "DUMP_ROWS", 5000)
    digest = 0xFEDCBA9876543210
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), _TableSource(t), None, digest)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == sorted(p.name for p in (tmp_path / "b").iterdir())
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    out = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(v.dtype == np.float64 for v in out.values())
    assert out["counts"].tolist() == [t.n_instances, t.n_distinct, t.n_buckets, t.n_kmers, len(t.read_ids)]
    assert (int(out["table_digest"][0]) << 32) | int(out["table_digest"][1]) == digest

    def full_or_rows(name, a):
        rows = out.get(f"{name}_rows")
        assert (rows is None) == (len(a) <= 5000)
        return a if rows is None else a[rows.astype(np.int64)]

    kc = full_or_rows("kmer_codes", t.kmer_codes.reshape(-1, t.kw))
    got = out["kmer_codes"].astype(np.uint64)
    assert got.shape == (len(kc), 2 * t.kw)
    for w in range(t.kw):
        np.testing.assert_array_equal((got[:, 2 * w] << np.uint64(32)) | got[:, 2 * w + 1], kc[:, w])
    for name, a in (("mmer_codes", t.mmer_codes), ("mmer_kmer_off", t.mmer_kmer_off), ("kmer_id_off", t.kmer_id_off),
                    ("read_ids", t.read_ids)):
        np.testing.assert_array_equal(out[name], full_or_rows(name, a).astype(np.float64))
