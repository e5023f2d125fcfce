"""Full-size bit-exact parity with the reference hot path: the table of the CUDA path dumped by gbin_table_dump against the
reference's process_read loop + prune_data over the whole input — md5 of the LC_ALL=C-sorted lines ("<mmer> <kmer> <id> <id> ...").
The reads are synthetic and seeded, so the expected md5 of every case is stored in tests/golden/fullsize_pins.json, whose
"produced_by" says which program dumped it (tests/golden/make_fullsize_pins.py: the unmodified reference binary when it is
built, else the oracle that tests/test_oracle_pins.py pins against the reference's dumps of the golden fixtures).  Where the
reference binary is built (oracle/build_ref.sh, from the reference's own sources), its dump of the same reads is compared too.
Sizes: BASELINE config 2 in full (the bench configuration), and the shapes of configs 4 and 5 on a prefix of their read stream."""
import ctypes as C
import json
import os
import subprocess

import pytest

import oracle_lib as O
from genome_assembly_b200 import binding as B
from genome_assembly_b200 import synth

pytestmark = pytest.mark.gpu

REF_DIR = os.path.join(O.ROOT, "oracle", "_ref")
with open(os.path.join(O.GOLDEN, "fullsize_pins.json")) as _f:
    PINS = {c["name"]: c for c in json.load(_f)["cases"]}


def sorted_md5(cmd_or_path, from_cmd: bool) -> str:
    env = dict(os.environ, LC_ALL="C")
    if from_cmd:
        p1 = subprocess.Popen(cmd_or_path, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
        p2 = subprocess.Popen(["sort", "-S", "2G"], stdin=p1.stdout, stdout=subprocess.PIPE, env=env)
    else:
        p1 = None
        p2 = subprocess.Popen(["sort", "-S", "2G", cmd_or_path], stdout=subprocess.PIPE, env=env)
    p3 = subprocess.run(["md5sum"], stdin=p2.stdout, capture_output=True, check=True)
    p2.wait()
    if p1 is not None:
        assert p1.wait() == 0
    assert p2.returncode == 0
    return p3.stdout.split()[0].decode()


def run_case(tmp_path, name, pipelines=(3,)):
    import torch
    assert torch.cuda.is_available()
    case = PINS[name]
    K, M, L, cutoff = case["k"], case["m"], case["read_len"], case["cutoff"]
    rs = synth.generate(case["n_reads"], L, error_rate=case["error_rate"], seed=case["seed"], starts=case["starts"])
    want = case["md5"]
    exe = os.path.join(REF_DIR, f"ref_K{K}_M{M}_C{cutoff}_R{L + 2}")
    if os.path.exists(exe):
        reads = tmp_path / "reads.txt"
        rs.buf.tofile(str(reads))
        assert sorted_md5([exe, str(reads)], True) == want, "the reference binary's dump differs from the stored pin"
    L_ = B.load_library()
    for pl in pipelines:
        b = B.Binner(K, M, cutoff, pipeline=pl)
        t = b.bin_host_raw(B.Binner._reads(rs.buf, rs.buf.size, rs.n_reads, stride=rs.stride, read_len=rs.read_len))
        assert b.pipeline_info()["last_used"] == pl, b.pipeline_info()
        assert t.n_kmers == case["surviving_kmers"], (pl, t.n_kmers, case["surviving_kmers"])
        dump = tmp_path / f"gpu_p{pl}.dump"
        assert L_.gbin_table_dump(C.byref(t), str(dump).encode()) == 0
        got = sorted_md5(str(dump), False)
        os.unlink(dump)
        b.close()
        assert got == want, (pl, got, want)


def test_full_cfg2_equals_the_reference_binary(tmp_path):
    """BASELINE config 2, all 1 M reads x 100 bp (70 M k-mer instances): the bench configuration, bit for bit."""
    run_case(tmp_path, "full_cfg2", pipelines=(3, 2))


def test_cfg4_shape_k63_equals_the_reference_binary(tmp_path):
    """Config 4's shape (K=63: 128-bit codes, M=15) on 200 000 x 250 bp (37.6 M instances)."""
    run_case(tmp_path, "cfg4_shape_k63")


def test_cfg5_shape_prune_heavy_equals_the_reference_binary(tmp_path):
    """Config 5's shape (K=25, M=9, 5 % substitutions) on 500 000 x 150 bp (63 M instances): m-mer buckets of tens of thousands of
    instances, so the extended keys, the spans and the global sort of pipeline 3 are all on the path."""
    run_case(tmp_path, "cfg5_shape_prune_heavy")
