"""The multi-GPU entry point of the C ABI (gbin_multi_*) driven by a plain C program — no Python in the data path, no torch, no
NCCL: tools/multi_demo.c bins a fixture on every GPU of the box (1 works too) and prints the sum of the owners' table digests,
which must equal the digest pinned for the fixture (derived from the unmodified reference binary's table).  fuzz_polyA and a
homopolymer batch overflow a shared-memory unit of the super-k-mer path: the call redoes the batch in instance-record form."""
import gzip
import json
import os
import subprocess

import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

DEMO = os.path.join(O.ROOT, "tools", "multi_demo")


def homopolymer_case(path):
    """3 000 reads of 100 A: one k-mer with 210 000 instances, more than a shared-memory unit holds.  Every GPU redoes its shard in
    instance-record form; the expected sizes and digest are the oracle's."""
    data = (b"A" * 100 + b"\n") * 3000
    path.write_bytes(data)
    starts, lens = O.fgets_split(data, 102)
    want = O.run(data, starts, lens, 31, 4, 1)
    return dict(k=31, m=4, cutoff=1, read_length_define=102, instances=int(want.n_instances), surviving_kmers=want.n_kmers,
                surviving_buckets=want.n_buckets, digest="%016x" % O.table_digest(want))


@pytest.mark.parametrize("name", ["cfg2_small", "cfg5_small", "cfg4_small", "cfg1_reads", "fuzz_polyA", "poly_a_3000"])
def test_c_program_bins_on_all_gpus_and_matches_the_pinned_digest(name, tmp_path):
    assert os.path.exists(DEMO), "tools/multi_demo is built by genome-assembly_b200/Makefile"
    path = tmp_path / "reads.txt"
    if name == "poly_a_3000":
        case = homopolymer_case(path)
    else:
        case = next(c for c in O.load_pins() if c["name"] == name)
        path.write_bytes(gzip.open(os.path.join(O.GOLDEN, case["file"]), "rb").read())
    p = subprocess.run([DEMO, str(path), str(case["k"]), str(case["m"]), str(case["cutoff"]), str(case["read_length_define"])],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    out = json.loads(p.stdout.strip().splitlines()[-1])
    assert out["gpus"] >= 1
    assert out["instances"] == case["instances"] and out["surviving_kmers"] == case["surviving_kmers"]
    assert out["buckets"] == case["surviving_buckets"]
    assert out["digest"] == case["digest"], out
