#!/usr/bin/env python
"""Generates tests/golden/fullsize_pins.json: the md5 of the LC_ALL=C-sorted table dump ("<mmer> <kmer> <ids...>" per line)
of each full-size case of tests/test_gpu_fullsize.py.

The reads are synthetic (genome_assembly_b200.synth, seeded), so only the md5 of the table has to be stored.  Every case is
dumped by the string-faithful oracle (oracle/_build/gbin_oracle_cli --strings), the restatement of the reference hot path that
tests/test_oracle_pins.py pins against the reference binary's own dumps of the golden fixtures, and by the code-space oracle
(the same CLI without --strings); the two must agree.  When the unmodified reference binary is built
(oracle/_ref/ref_K*_M*_C*_R*, by oracle/build_ref.sh from the reference's own sources) it dumps the case too, the oracle must
agree with it, and the pin says so in "produced_by".  CPU only; the cfg2 case takes a few minutes:
    make -C oracle && python tests/golden/make_fullsize_pins.py
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from genome_assembly_b200 import synth  # noqa: E402

CLI = os.path.join(ROOT, "oracle", "_build", "gbin_oracle_cli")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")

# (name, n_reads, read_len, K, M, error_rate, starts); cutoff 1, genome and reads from seed 20
CASES = [
    ("full_cfg2", 1_000_000, 100, 31, 11, 0.01, "triangular"),
    ("cfg4_shape_k63", 200_000, 250, 63, 15, 0.01, "uniform"),
    ("cfg5_shape_prune_heavy", 500_000, 150, 25, 9, 0.05, "uniform"),
]


def sorted_md5(cmd):
    """md5 and line count of the LC_ALL=C-sorted stdout of cmd."""
    env = dict(os.environ, LC_ALL="C")
    p1 = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    p2 = subprocess.Popen(["sort", "-S", "2G"], stdin=p1.stdout, stdout=subprocess.PIPE, env=env)
    p1.stdout.close()
    h, lines = hashlib.md5(), 0
    for chunk in iter(lambda: p2.stdout.read(1 << 20), b""):
        h.update(chunk)
        lines += chunk.count(b"\n")
    assert p1.wait() == 0 and p2.wait() == 0
    return h.hexdigest(), lines


def main():
    pins = []
    for name, n, L, K, M, err, starts in CASES:
        rs = synth.generate(n, L, error_rate=err, seed=20, starts=starts)
        exe = os.path.join(REF_DIR, f"ref_K{K}_M{M}_C1_R{L + 2}")
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "reads.txt")
            rs.buf.tofile(path)
            args = [CLI, path, str(K), str(M), "1", str(L + 2)]
            md5, lines = sorted_md5(args + ["--strings"])
            assert sorted_md5(args) == (md5, lines), name
            if os.path.exists(exe):
                assert sorted_md5([exe, path]) == (md5, lines), f"{name}: the oracle differs from the reference binary"
                produced_by = "the unmodified reference binary, and the oracle agrees"
            else:
                produced_by = "the oracle (string-faithful and code-space modes agree); the reference binary was not built"
        pin = dict(name=name, n_reads=n, read_len=L, k=K, m=M, cutoff=1, error_rate=err, starts=starts, seed=20,
                   read_length_define=L + 2, md5=md5, surviving_kmers=lines, produced_by=produced_by)
        pins.append(pin)
        print(pin, flush=True)
    with open(os.path.join(HERE, "fullsize_pins.json"), "w") as f:
        json.dump(dict(generated_by="tests/golden/make_fullsize_pins.py",
                       sort="LC_ALL=C sort of dump lines, md5 of the result", cases=pins), f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
