"""Pipeline 3's 1024-instance grouping kernel, where a pair of warps works on one unit, against the oracle.

The read set covers a 40 kb genome about 75 times, so that with plain m-mer keys (K=31, M=11) many buckets hold 513-1024
instances (each one a unit of its own, grouped by the large-unit launch) and some hold more than 1024 (atoms cut into d-rounds,
grouped by the same launch without the per-entry tables).  K=63 at capacity 1024 runs the single-launch form of the same kernel,
whose units pack many buckets."""
import numpy as np
import pytest

import oracle_lib as O
from genome_assembly_b200 import binding as B
from genome_assembly_b200 import synth

L = 100


def deep_reads():
    rs = synth.generate(30000, L, genome_len=40000, seed=7)
    starts = np.arange(rs.n_reads, dtype=np.uint64) * rs.stride
    lens = np.full(rs.n_reads, rs.read_len, dtype=np.uint32)
    return rs, starts, lens


def test_fixture_has_pair_sized_buckets_and_rounds():
    """The read set reaches both paths of the pair kernel: buckets of 513-1024 instances and buckets above 1024."""
    rs, starts, lens = deep_reads()
    tup, _ = O.scan_all(rs.as_bytes(), starts, lens, 31, 11)
    _, c = np.unique(tup["mmer"], return_counts=True)
    assert ((c > 512) & (c <= 1024)).sum() >= 1000, np.bincount(np.minimum(c // 256, 8))
    assert (c > 1024).sum() >= 50, c.max()


@pytest.mark.gpu
@pytest.mark.parametrize("K,M,cap", [(31, 11, 0), (63, 15, 1024)])
@pytest.mark.parametrize("cutoff", [1, 0])
def test_pair_grouping_equals_the_oracle(K, M, cap, cutoff):
    import torch
    assert torch.cuda.is_available()
    rs, starts, lens = deep_reads()
    b = B.Binner(K, M, cutoff, pipeline=3)
    if cap:
        b.set_tuning("v3_cap", cap)
    b.set_kernel_profiling(True)
    got = b.bin_host(rs.buf, rs.n_reads, stride=rs.stride, read_len=rs.read_len)
    want = O.run(rs.as_bytes(), starts, lens, K, M, cutoff)
    for name in ("mmer_codes", "mmer_kmer_off", "kmer_codes", "kmer_id_off", "read_ids"):
        np.testing.assert_array_equal(getattr(got, name), getattr(want, name).reshape(-1), err_msg=name)
    info, st, prof = b.pipeline_info(), b.run_stats(), b.kernel_profile()
    assert info["last_used"] == 3 and info["fallbacks"] == 0, info
    assert st["key_nc"] == 1, st  # plain m-mer keys: capacity 1024
    # the grouping was launched in the expected form (the large-unit and the small-unit launch side by side for K <= 32, one launch
    # otherwise); that the pair kernel grouped its units correctly is shown by the comparison with the oracle above, since the
    # fixture's 513-1024-instance buckets and d-round units can only be grouped by it
    launches = prof["skr_group"]["launches"]
    if cap == 0:
        assert launches >= 2 and launches % 2 == 0, prof["skr_group"]
    else:
        assert launches >= 1, prof["skr_group"]
    b.close()
