#!/usr/bin/env python
"""bench.py — canonical k-mers binned+pruned per second on B200 (BASELINE.json metric).

A step = one pass of the hot path (process_read over every read -> two-level grouping -> prune)
over one batch of synthetic reads.  N=1: BASELINE config 2 (1 M reads x 100 bp, K=31, M=11, 1 %
substitutions, generate_reads.py's triangular start walk).  N>1: BASELINE config 3 (100 M reads x 150 bp, the configuration
north_star names for 2/4/8 GPUs), strong scaling: one read set (the same at every N: it is drawn block by block from one
genome, every block with its own generator) is split evenly over the ranks by contiguous ranges, records are exchanged by
m-mer owner (peer stores over NVLink), every rank groups the buckets it owns.  The sum of the owners' table digests is
printed and checked against profiles/expected_digests.json: it must be the same at every N.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  `value` is device-resident throughput (inputs in HBM when the
timed region starts), `e2e` goes through the public host-buffer call (pinned H2D + pipeline + D2H of
the table inside the timed region), `roofline` is the dominant kernel class (the shared-memory grouping kernel) timed
live with CUDA events on its launching stream, `cpu_baseline` is the UNMODIFIED reference binary
(oracle/_ref) on one host core over a bounded prefix of the same reads.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "canonical k-mers binned+pruned per second"
UNIT = "k-mers/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gbin", choices=["gbin", "reference"])
    ap.add_argument("--workload", default="auto", help="cfg2..cfg5; auto = cfg2 on one GPU, cfg3 on several")
    ap.add_argument("--no-selftest", action="store_true", help="N > 1: skip the sharded run of the golden fixtures before the timed region")
    ap.add_argument("--reads-per-gpu", type=int, default=0, help="override the workload's read count (debug)")
    ap.add_argument("--scaling", default="auto", choices=["auto", "weak", "strong"],
                    help="weak: every GPU holds the workload's read count (default for cfg2); strong: the workload's reads are split "
                         "over the GPUs (default for cfg3-5, whose BASELINE sizes are totals)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU record exchange: peer = partition kernel stores into the owners' buffers over NVLink (default), nccl = all_to_all_single")
    ap.add_argument("--e2e-contexts", type=int, default=2, help="contexts (= host threads) of the --e2e-overlapped leg")
    ap.add_argument("--no-e2e-overlapped", action="store_true", help="skip the two-context leg of e2e (e2e.value is then the single-call figure)")
    ap.add_argument("--e2e-overlapped", action="store_true", help="(default now; kept so that older command lines still parse)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the table of the last timed step as DIR/<name>.npy (float64, see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's table; --impl reference computes none")
    return a


READ_BLOCK = 250_000  # reads per generator block of the strong-scaling read sets


def workload_params(name, reads_override=0, scaling="auto", world=1):
    """Per-GPU shape of the workload.  weak: n_reads per GPU = the workload's count; strong: the count is split."""
    from genome_assembly_b200 import synth
    if name == "auto":
        name = "cfg2" if world == 1 else "cfg3"
    w = dict(synth.WORKLOADS[name])
    w["name"] = name
    if scaling == "auto":
        scaling = "weak" if name == "cfg2" else "strong"
    w["scaling"] = scaling
    w["total_reads"] = w["n_reads"] * world if scaling == "weak" else w["n_reads"]
    if scaling == "strong":
        w["n_reads"] = w["n_reads"] // world
    if reads_override:
        w["n_reads"] = reads_override
        w["total_reads"] = reads_override * world
    return w


def make_reads(w, rank, world):
    """This rank's shard: config-shaped reads from one shared genome (30x coverage over all ranks' reads).  Strong scaling with
    uniform starts: the whole read set is a sequence of READ_BLOCK-sized blocks, block b drawn with a generator seeded by b,
    and rank r holds a contiguous range of blocks — the same read set, in the same order, at every N."""
    import numpy as np
    from genome_assembly_b200 import synth
    n = w["n_reads"]
    glen = synth.default_genome_len(w["total_reads"], w["read_len"])
    blocked = w["scaling"] == "strong" and w["starts"] == "uniform" and w["total_reads"] % (READ_BLOCK * world) == 0
    w["read_set"] = f"blocks of {READ_BLOCK} reads, one generator per block: identical at every GPU count" if blocked else "one generator per rank"
    if not blocked:
        return synth.generate(n, w["read_len"], genome_len=glen, error_rate=w["error_rate"], seed=20, read_seed=20 + rank, starts=w["starts"])
    stride = w["read_len"] + 1
    b0 = rank * (n // READ_BLOCK)
    try:
        import torch
        cuda = torch.cuda.is_available()
    except ImportError:
        cuda = False
    if cuda:  # drawn on the GPU: seconds instead of minutes for the 100 M-read configurations
        w["read_set"] += "; drawn on the GPU (torch generators)"
        d = synth.blocked_reads_torch(glen, n // READ_BLOCK, b0, READ_BLOCK, w["read_len"], error_rate=w["error_rate"], seed=20,
                                      device=torch.device("cuda", torch.cuda.current_device()))
        buf = d.cpu().numpy()
        del d
        torch.cuda.empty_cache()
        return synth.ReadSet(buf=buf, n_reads=n, read_len=w["read_len"], stride=stride, genome_len=glen, seed=20, error_rate=w["error_rate"],
                             starts_kind="uniform")
    w["read_set"] += "; drawn on the host (numpy generators)"
    genome = synth.make_genome(glen, 20)
    buf = np.empty(n * stride, dtype=np.uint8)
    for k in range(n // READ_BLOCK):
        synth.reads_from_genome(genome, READ_BLOCK, w["read_len"], error_rate=w["error_rate"], read_seed=b0 + k,
                                out=buf[k * READ_BLOCK * stride:(k + 1) * READ_BLOCK * stride])
    return synth.ReadSet(buf=buf, n_reads=n, read_len=w["read_len"], stride=stride, genome_len=glen, seed=20, error_rate=w["error_rate"],
                         starts_kind="uniform")


# ------------------------------------------------------------------------------------------ CPU reference leg

def ref_binary(w, makefile_flags=False):
    """-O2 build of the unmodified reference by default; makefile_flags: the build the reference's makefile makes (-g, no optimisation)."""
    name = f"ref_K{w['k']}_M{w['m']}_C{w['cutoff']}_R{w['read_len'] + 2}" + ("_O0" if makefile_flags else "")
    return os.path.join(ROOT, "oracle", "_ref", name)


def time_reference(w, rs, n_sample_reads, makefile_flags=False):
    """Times the reference's own process_read loop + prune_data (binning.c:1158-1169) on the first
    n_sample_reads reads of the shard; returns (k-mers/s, dict)."""
    exe = ref_binary(w, makefile_flags)
    n = min(n_sample_reads, rs.n_reads)
    inst = n * (rs.read_len - w["k"] + 1)
    with tempfile.NamedTemporaryFile(suffix=".txt", delete=False) as tf:
        tf.write(rs.buf[: n * rs.stride].tobytes())
        path = tf.name
    try:
        if os.path.exists(exe):
            p = subprocess.run([exe, path, "--time"], capture_output=True, text=True, check=True)
            st = json.loads(p.stdout.strip().splitlines()[-1])
            secs = st["process_s"] + st["prune_s"]
            assert st["instances"] == inst
            kind = "reference"
        else:  # the reference could not be built here: fall back to the oracle port (still CPU, still 1 thread)
            cli = os.path.join(ROOT, "oracle", "_build", "gbin_oracle_cli")
            p = subprocess.run([cli, path, str(w["k"]), str(w["m"]), str(w["cutoff"]), str(w["read_len"] + 2), "--time"],
                               capture_output=True, text=True, check=True)
            st = json.loads(p.stdout.strip().splitlines()[-1])
            secs = st["total_s"]
            kind = "port"
    finally:
        os.unlink(path)
    return inst / secs, dict(kind=kind, cores=1, seconds=secs, instances=inst,
                             sample=f"first {n} reads of the rank-0 shard ({inst} k-mer instances), process_read loop + prune_data, 1 thread (the reference is single-threaded and non-reentrant, binning.c:300-303)")


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    w = workload_params(a.workload, a.reads_per_gpu, a.scaling, max(a.gpus, 1))
    if w["scaling"] == "strong" and w["n_reads"] > READ_BLOCK and w["n_reads"] % READ_BLOCK == 0:
        w["n_reads"] = READ_BLOCK  # the sample is a prefix of rank 0's shard: its first generator block is enough
    rs = make_reads(w, 0, max(a.gpus, 1))
    sample_reads = min(w["n_reads"], 200_000 if w["read_len"] <= 100 else 100_000)  # the cpu_baseline sample: ~14 M instances, ~9 s per step
    for _ in range(a.warmup):
        time_reference(w, rs, sample_reads)
    vals, info = [], None
    t0 = time.perf_counter()
    for _ in range(a.steps):
        v, info = time_reference(w, rs, sample_reads)
        vals.append(v)
    wall = time.perf_counter() - t0
    inst = info["instances"]
    value = inst * a.steps / sum(inst / v for v in vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * wall / max(a.steps, 1), "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
        "dtype": "u64" if w["k"] <= 32 else "u128", "data": "synthetic",
        "config": config_dict(a, w, max(a.gpus, 1)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ helpers

def config_dict(a, w, world):
    return {"workload": f"{w['name']}: {w['n_reads']} reads x {w['read_len']} bp per GPU ({w['total_reads']} in total, {w['scaling']} scaling), "
                        f"K={w['k']}, M={w['m']}, cutoff={w['cutoff']}, {w['error_rate'] * 100:g}% substitutions, {w['starts']} starts, "
                        f"genome {w['total_reads'] * w['read_len'] // 30} bp",
            "read_set": w.get("read_set"),
            "k": w["k"], "m": w["m"], "cutoff": w["cutoff"], "reads_per_gpu": w["n_reads"], "read_len": w["read_len"],
            "parallelism": f"reads split evenly over {world} GPU(s); records exchanged by owner = hash(mmer) -> [0, {world})" if world > 1 else "single GPU",
            "l2": "L2 flushed (256 MiB memset) before every timed step; per-step device times summed"}


def sharded_selftest(B, g, dist, torch, dev, rank, world, local, exchange):
    """Collective.  The golden fixtures go through the multi-GPU path (reads split by contiguous ranges, records exchanged by
    owner, every rank groups its buckets); the sum of the owners' digests must equal the digest pinned in tests/golden/pins.json
    (derived from the unmodified reference binary's dump).  Raises on a mismatch."""
    import gzip
    import numpy as np
    from genome_assembly_b200.dist import GpuStages, ShardedBinner
    pins = json.load(open(os.path.join(ROOT, "tests", "golden", "pins.json")))["cases"]
    done = []
    for name in ("cfg2_small", "cfg3_small", "cfg5_small"):
        case = next(c for c in pins if c["name"] == name)
        data = gzip.open(os.path.join(ROOT, "tests", "golden", case["file"]), "rb").read()
        with tempfile.NamedTemporaryFile(suffix=".txt", delete=False) as tf:
            tf.write(data)
        try:
            buf, starts, lens = B.read_file_fgets(tf.name, case["read_length_define"])
        finally:
            os.unlink(tf.name)
        n = len(starts)
        lo, hi = (n * rank) // world, (n * (rank + 1)) // world
        b = g.Binner(case["k"], case["m"], case["cutoff"], device=local)
        d = torch.from_numpy(np.frombuffer(buf, dtype=np.uint8).copy()).to(dev)
        st_ = torch.from_numpy(starts[lo:hi].astype(np.int64)).to(dev)
        ln_ = torch.from_numpy(lens[lo:hi].astype(np.int32)).to(dev)
        rd = B.Binner._reads(d, d.numel(), hi - lo, starts=st_, lens=ln_)
        sb = ShardedBinner(GpuStages(b), exchange=exchange)
        t = sb.run(rd, arrival_base=lo)
        dg = b.table_digest(t, B.stream_handle(torch.cuda.current_stream()))
        tot = torch.tensor([dg - (1 << 64) if dg >= (1 << 63) else dg], dtype=torch.int64, device=dev)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        got = "%016x" % (int(tot[0]) & ((1 << 64) - 1))
        if got != case["digest"]:
            raise SystemExit(f"bench.py selftest: {name} over {world} GPUs gives digest {got}, the reference's table has {case['digest']}")
        done.append(name)
        dist.barrier()
        b.close()
    return {"cases": done, "world": world, "result": "digests equal the reference-derived pins"}


class ClockSampler:
    """nvidia-smi sampled every 20 ms from process start; only samples whose timestamp falls inside the marked
    window (warm-up + timed region) are used, and of those the loaded (upper) half for the median SM clock."""
    QUERY = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.tf = tempfile.NamedTemporaryFile(suffix=".csv", delete=False)
        self.proc = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=self.tf, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tf.close()
        rows = []
        with open(self.tf.name) as f:
            for ln in f:
                p = [x.strip() for x in ln.split(",")]
                if len(p) < 10:
                    continue
                try:
                    ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    rows.append((ts, float(p[2]), float(p[3]), p[6:10]))
                except ValueError:
                    continue
        os.unlink(self.tf.name)
        inside = [r for r in rows if self.t0 is not None and self.t0 - 0.02 <= r[0] <= (self.t1 or 1e18) + 0.02]
        use = inside if inside else rows
        if use:
            sm = sorted(r[1] for r in use)
            reasons = set()
            for r in use:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            out.update(sm_mhz=statistics.median(sm[len(sm) // 2:]), sm_max_mhz=max(r[2] for r in use), reasons=sorted(reasons),
                       samples=len(use), samples_total=len(rows), window="warm-up + timed region" if inside else "whole process")
        return out


DUMP_ROWS = 1 << 18  # rows kept per dumped array; longer arrays are sampled


def dump_outputs(out_dir, binner, table, digest, suffix=""):
    """Writes the pruned table of the last timed step as float64 .npy files, so that two builds can be compared output for
    output: counts.npy (n_instances, n_distinct, n_buckets, n_kmers, n_ids), table_digest.npy (gbin_table_digest, which
    covers the whole table), and the table's arrays mmer_codes, mmer_kmer_off, kmer_codes, kmer_id_off and read_ids.  64-bit
    codes are split into 32-bit limbs, most significant first, so that float64 holds them exactly: kmer_codes has
    2 * kmer_words columns.  An array longer than DUMP_ROWS rows is cut to a fixed, seeded sample of DUMP_ROWS rows, whose
    indices go to <name>_rows.npy.  At most about 26 MiB in all."""
    import numpy as np
    h = binner.table_to_host(table)
    os.makedirs(out_dir, exist_ok=True)

    def limbs(x):
        x = np.asarray(x, dtype=np.uint64)
        return np.stack([x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)], axis=-1).reshape(len(x), 2)

    def save(name, a):
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.ascontiguousarray(a, dtype=np.float64))

    save("counts", [h.n_instances, h.n_distinct, h.n_buckets, h.n_kmers, h.n_ids])
    save("table_digest", limbs([digest])[0])
    arrays = {"mmer_codes": h.mmer_codes, "mmer_kmer_off": h.mmer_kmer_off, "kmer_codes": limbs(h.kmer_codes).reshape(h.n_kmers, 2 * h.kw),
              "kmer_id_off": h.kmer_id_off, "read_ids": h.read_ids}
    for name, a in arrays.items():
        assert a.dtype != np.uint64 or a.size == 0 or int(a.max()) < (1 << 53), name  # exact in float64
        if len(a) > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(len(a), DUMP_ROWS, replace=False))
            save(f"{name}_rows", rows)
            a = a[rows]
        save(name, a)


_REAL_STDOUT = None


def emit(line: dict):
    """The one JSON line goes to the process's original stdout; everything else that libraries print on fd 1 (NCCL's
    version banner, for instance) is diverted to stderr so that the driver can parse stdout as a single line."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    a = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference_arm(a)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import genome_assembly_b200 as g
    from genome_assembly_b200.dist import GpuStages, ShardedBinner

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the binning path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()  # nvidia-smi takes about a second to deliver its first sample: start it before the data is generated
    w = workload_params(a.workload, a.reads_per_gpu, a.scaling, world)
    K, M, cutoff = w["k"], w["m"], w["cutoff"]
    rs = make_reads(w, rank, world)
    W = rs.read_len - K + 1
    n_inst_rank = rs.n_reads * W
    n_inst_total = n_inst_rank * world

    binner = g.Binner(K, M, cutoff, device=local)
    B = g.binding
    # host copy in pinned memory (e2e leg) and device-resident copy (value leg)
    h_reads = torch.from_numpy(rs.buf).pin_memory()
    d_reads = h_reads.to(dev, non_blocking=True)
    torch.cuda.synchronize()
    stream = B.stream_handle(torch.cuda.current_stream())
    rd_dev = B.Binner._reads(d_reads, d_reads.numel(), rs.n_reads, stride=rs.stride, read_len=rs.read_len, id_base=rank * rs.n_reads)
    rd_host = B.Binner._reads(h_reads, h_reads.numel(), rs.n_reads, stride=rs.stride, read_len=rs.read_len, id_base=rank * rs.n_reads)

    # ---- N > 1: before anything is timed, the sharded path must reproduce the pinned digests of the golden fixtures
    selftest = None
    if world > 1 and not a.no_selftest:
        selftest = sharded_selftest(B, g, dist, torch, dev, rank, world, local, a.exchange)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    stages = GpuStages(binner)
    sharded = ShardedBinner(stages, time_stages=True, exchange=a.exchange) if world > 1 else None
    stage_ms = {"scan": 0.0, "partition": 0.0, "exchange": 0.0, "group": 0.0}

    def step_device():
        if world == 1:
            return binner.bin_device_raw(rd_dev, stream)
        return sharded.run(rd_dev, arrival_base=rank * rs.n_reads)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if sampler:
        sampler.mark_begin()

    # ---- warm-up (also sizes every workspace buffer)
    table = None
    for _ in range(max(a.warmup, 0)):
        table = step_device()
    barrier()

    # ---- timed region: K steps, L2 flushed before each, device time per step from CUDA events
    binner.set_kernel_profiling(True)
    launches = 0
    launches_before = stages.launches
    barrier()
    t_wall0 = time.perf_counter()
    step_ms = []
    for _ in range(a.steps):
        flush.zero_()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        table = step_device()
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
        launches += binner.timings()["kernel_launches"] if world == 1 else 0
        if sharded is not None:
            st_ = sharded.stats
            for k_, v_ in (("scan", st_.scan_ms), ("partition", st_.partition_ms), ("exchange", st_.exchange_ms), ("group", st_.group_ms)):
                stage_ms[k_] += v_ / a.steps
    barrier()
    wall_s = time.perf_counter() - t_wall0
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    prof = binner.kernel_profile()
    binner.set_kernel_profiling(False)
    if world > 1:
        launches = stages.launches - launches_before
    total_ms = float(sum(step_ms))
    tms = torch.tensor([total_ms, float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = tms.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tms.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_ms = float(mx[0])
        launches = int(sm[1])
    value = n_inst_total * a.steps / (total_ms / 1e3)

    # ---- table stats of the last step (sanity: work was really done)
    stats = {"instances": int(table.n_instances), "distinct": int(table.n_distinct), "surviving_kmers": int(table.n_kmers),
             "surviving_ids": int(table.n_ids), "buckets": int(table.n_buckets)}
    # ---- digest of the whole job's table: the sum (mod 2^64) of the owners' digests; the same at every GPU count for a strong-scaling read set
    dg = binner.table_digest(table, stream)
    tot = torch.tensor([dg - (1 << 64) if dg >= (1 << 63) else dg, stats["instances"], stats["surviving_kmers"], stats["surviving_ids"]],
                       dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)  # two's-complement wrap-around = addition modulo 2^64
    digest = "%016x" % (int(tot[0]) & ((1 << 64) - 1))
    job = {"instances": int(tot[1]), "surviving_kmers": int(tot[2]), "surviving_ids": int(tot[3])}
    dkey = f"{w['name']}:{w['total_reads']}x{w['read_len']}:K{K}:M{M}:C{cutoff}:{'blocks' if 'blocks' in w.get('read_set', '') else 'ranks'}:{'gpu' if 'GPU' in w.get('read_set', '') else 'host'}"
    expected = None
    try:
        expected = json.load(open(os.path.join(ROOT, "profiles", "expected_digests.json"))).get(dkey)
    except (OSError, ValueError):
        pass
    digest_info = {"table_digest": digest, "key": dkey, "expected": expected, "ok": (digest == expected) if expected else None,
                   "what": "gbin_table_digest: order-independent hash of every (m-mer, k-mer, ordered id list), summed over the owners"}
    if expected and digest != expected and rank == 0:
        print(f"bench.py: table digest {digest} differs from profiles/expected_digests.json[{dkey}] = {expected}", file=sys.stderr)
    if a.dump_outputs:  # before the e2e leg, which reuses the context's buffers that hold the device table
        dump_outputs(a.dump_outputs, binner, table, dg, f"_rank{rank}" if world > 1 else "")

    # ---- e2e: public host-buffer call, pinned H2D + pipeline + D2H of the table inside the timed region
    e2e = None
    if not a.no_e2e and world == 1:
        for _ in range(2):
            binner.bin_host_raw(rd_host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(a.steps):
            t = binner.bin_host_raw(rd_host)
            d2h = int(t.n_kmers * (8 * t.kmer_words + 8) + 8 + t.n_ids * 4 + t.n_buckets * 12 + 8)
        e2e_s = time.perf_counter() - t0
        e2e = {"value": n_inst_total * a.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h_reads.numel()),
               "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / a.steps, "timing": "host wall clock around gbin_bin_reads_host",
               "stage_ms_last_step": binner.timings()}
        if not a.no_e2e_overlapped:
            # two contexts, two host threads (ctypes releases the GIL inside the C call): every batch still pays its own H2D and
            # D2H inside the timed region, but the copies of consecutive batches overlap
            import threading
            extra = [g.Binner(K, M, cutoff, device=local) for _ in range(max(a.e2e_contexts, 2) - 1)]
            group = [binner] + extra
            for bb in group:
                bb.bin_host_raw(rd_host)
            torch.cuda.synchronize()
            per_thread = a.steps

            def worker(bb):
                for _ in range(per_thread):
                    bb.bin_host_raw(rd_host)
            ths = [threading.Thread(target=worker, args=(bb,)) for bb in group]
            t0 = time.perf_counter()
            for th in ths:
                th.start()
            for th in ths:
                th.join()
            ov_s = time.perf_counter() - t0
            nb = len(group) * per_thread
            e2e["overlapped"] = {"value": n_inst_total * nb / ov_s, "unit": UNIT, "batches": nb, "contexts": len(group),
                                 "ms_per_batch": 1e3 * ov_s / nb,
                                 "how": "one context per host thread, each batch with its own pinned H2D and table D2H"}
            for bb in extra:
                bb.close()
            # the headline end-to-end figure is the pipelined one (what a caller with a stream of batches gets: every batch
            # still pays its whole H2D and D2H inside the timed region); the one-call-at-a-time figure stays beside it
            e2e["single_call"] = {"value": e2e["value"], "ms_per_step": e2e["ms_per_step"], "timing": e2e["timing"]}
            e2e["value"] = e2e["overlapped"]["value"]
            e2e["ms_per_step"] = e2e["overlapped"]["ms_per_batch"]
            e2e["timing"] = ("host wall clock over %d gbin_bin_reads_host calls issued from %d host threads, one context each (PCIe is full duplex: "
                             "the H2D of one batch overlaps the D2H of the other); single_call = the same call issued one at a time"
                             % (nb, len(group)))
    elif not a.no_e2e:
        # multi-GPU e2e: pinned H2D of every rank's shard + sharded pipeline + D2H of every owner table
        def e2e_step():
            d = h_reads.to(dev, non_blocking=True)
            rdx = B.Binner._reads(d, d.numel(), rs.n_reads, stride=rs.stride, read_len=rs.read_len, id_base=rank * rs.n_reads)
            tb = sharded.run(rdx, arrival_base=rank * rs.n_reads)
            ht = binner.table_to_pinned_raw(tb, stream)
            return int(ht.n_kmers * (8 * ht.kmer_words + 8) + 8 + ht.n_ids * 4 + ht.n_buckets * 12 + 8)
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(a.steps):
            d2h = e2e_step()
        barrier()
        e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e = {"value": n_inst_total * a.steps / float(e2e_s[0]), "unit": UNIT, "h2d_bytes_per_step": int(h_reads.numel()) * world,
               "d2h_bytes_per_step": d2h * world, "ms_per_step": 1e3 * float(e2e_s[0]) / a.steps,
               "timing": "host wall clock, max over ranks; per rank: pinned H2D of its shard, sharded pipeline, D2H of its owner table into the pinned arena"}

    # ---- input side (SURVEY 8 row f2): main's fgets loop on the device over this rank's file image (the reads buffer IS the
    # file: one newline-terminated line per read), READ_LENGTH = L + 2 as for the synthetic configs
    input_split = None
    if world == 1 and not a.no_e2e:
        rd_split = binner.split_reads_device(d_reads, d_reads.numel(), rs.read_len + 2, stream)
        assert int(rd_split.n_reads) == rs.n_reads, (int(rd_split.n_reads), rs.n_reads)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ms = []
        for _ in range(5):
            flush.zero_()
            ev0.record()
            binner.split_reads_device(d_reads, d_reads.numel(), rs.read_len + 2, stream)
            ev1.record()
            ev1.synchronize()
            ms.append(ev0.elapsed_time(ev1))
        best = min(ms)
        alg = 2.0 * d_reads.numel() + 12.0 * rs.n_reads + 8.0 * rs.n_reads  # image read twice (count, emit), newline positions, starts + lens
        input_split = {"what": "gbin_split_reads_device: fgets-exact split of the file image into starts/lens on the device (includes its two host round trips)",
                       "ms": best, "reads": rs.n_reads, "bytes": int(d_reads.numel()), "achieved_GBps": alg / (best / 1e3) / 1e9,
                       "algorithmic_bytes": alg}

    # ---- roofline of the dominant kernel (the kernel class with the most device time in the timed region)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    rb = binner.record_bytes
    KW = 1 if K <= 32 else 2
    rstats = binner.run_stats()
    n_skr = rstats["n_super_kmers"]
    skr_b = binner.skr_record_bytes
    n_rec = stats["instances"]  # k-mer instances this rank grouped in the last step
    # algorithmic (compulsory) HBM bytes of ONE launch of each kernel class, see DESIGN.md section 4
    n_ent = n_skr * (rstats.get("key_nc", 1) or 1)
    out_bytes = stats["surviving_kmers"] * (8.0 * KW + 4 + 8) + 4.0 * stats["surviving_ids"]
    v3 = binner.pipeline_info()["last_used"] == 3
    alg_bytes = {
        "radix_scatter": (2.0 * 8 * n_ent if v3 else 2.0 * skr_b * n_skr) if n_skr else (2.0 * rb * n_rec),
        "radix_hist": (1.0 * 8 * n_ent if v3 else 1.0 * skr_b * n_skr) if n_skr else (1.0 * rb * n_rec),
        "scan_reads": float(h_reads.numel()) + rb * n_inst_rank,
        "skr_scan": float(h_reads.numel()) + skr_b * n_skr,
        # pipeline 3: entries + records read once, the unit's part of the table written once (to staging); pipeline 2: records + instance prefix in, table out
        "skr_group": ((8.0 * n_ent + skr_b * n_skr + out_bytes) if v3 else ((skr_b + 4.0) * n_skr + out_bytes)),
        "v3_entries": 32.0 * n_skr + 9.0 * n_ent,  # a 32-byte sector per record header, 8-byte entry + 1 byte per slot out
        "v3_span": 2.0 * out_bytes,                # finalize: staging -> final place
        "find_runs": 3.0 * rb * n_rec + 8.0 * n_rec,
    }
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu export of this build's kernels (profiles/ncu_traffic.json,
    # written by profiles/tools/ncu_traffic.py from an `ncu --set full` capture); null when there is no entry for the dominant kernel / workload
    ncu_traffic = {}
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if tj.get("workload") == w["name"] and world == 1 and not a.reads_per_gpu:
            ncu_traffic = {k: v["dram_bytes_per_launch"] for k, v in tj.get("kernels", {}).items()}
    except (OSError, ValueError, KeyError):
        pass
    roofline = None
    timed = {k: v for k, v in prof.items() if v["launches"] and k in alg_bytes}
    if timed:
        dom = max(timed, key=lambda k: timed[k]["ms"])
        sc = timed[dom]
        alg = alg_bytes[dom]
        # classes whose algorithmic bytes are stated per step but which take several launches per step (the grouping stage: two
        # launches share the unit list; multi-pass batches): bytes per launch = bytes per step / launches per step
        per_step_classes = ("skr_group", "v3_span", "skr_plan", "v3_entries", "skr_scan")
        if dom in per_step_classes and sc["launches"] > a.steps:
            alg = alg * a.steps / sc["launches"]
        avg_ms = sc["ms"] / sc["launches"]
        ach = alg / (avg_ms / 1e3) / 1e9
        pipe_bytes_per_inst = (rs.read_len + 1) / W + 2 * rb + 4  # SURVEY section 8(d)
        pipe_ach = pipe_bytes_per_inst * n_inst_rank * a.steps / (float(sum(step_ms)) / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_traffic.get(dom),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "launches": sc["launches"], "avg_launch_ms": avg_ms,
                    "share_of_step": sc["ms"] / float(sum(step_ms)),
                    "note": "HBM is not what bounds this kernel: it groups k-mers in shared memory (hash insert, ranks, survivor order), one warp per unit; "
                            "see DESIGN.md 4 and profiles/ for the ncu evidence",
                    "pipeline": {"algorithmic_bytes_per_kmer": pipe_bytes_per_inst, "achieved": pipe_ach, "frac": pipe_ach / peak,
                                 "note": "whole step against SURVEY 8(d)'s compulsory-traffic model (37.4 B per k-mer instance at cfg2)"},
                    "per_kernel_ms_per_step": {k: v["ms"] / a.steps for k, v in prof.items()},
                    "per_kernel_achieved_gbs": {k: alg_bytes[k] * (a.steps if k in per_step_classes else v["launches"]) / (v["ms"] / 1e3) / 1e9
                                                for k, v in timed.items() if v["ms"] > 0},
                    "run_stats": rstats, "pipeline_info": binner.pipeline_info()}

    # ---- CPU baseline (rank 0, N=1 only): the unmodified reference binary on one host core
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        try:
            v, info = time_reference(w, rs, 200_000)
            cpu = {"value": v, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"],
                   "seconds": info["seconds"], "host_cores_available": os.cpu_count(), "build": "-O2"}
            if os.path.exists(ref_binary(w, makefile_flags=True)):  # SURVEY 8(d): also with the reference makefile's own flags (-g)
                try:
                    v0, info0 = time_reference(w, rs, 50_000, makefile_flags=True)
                    cpu["value_makefile_flags"] = v0
                    cpu["makefile_flags_sample"] = f"first 50000 reads, built with -g as in the reference's makefile ({info0['seconds']:.1f} s)"
                except Exception as e:  # noqa: BLE001
                    cpu["makefile_flags_sample"] = f"unavailable: {type(e).__name__}: {e}"
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "unavailable", "sample": f"{type(e).__name__}: {e}"}

    # ---- the reference-named entry points (process_read x n + prune_data, as main drives them) on the cpu_baseline's sample: staging
    # of the reads, the GPU path, and the ZHashTable / ll_node graph the reference's iterators walk (VERDICT r1 item 9)
    shim = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        exe = os.path.join(ROOT, "tools", "shim_bench")
        try:
            n = min(200_000, rs.n_reads)
            with tempfile.NamedTemporaryFile(suffix=".txt", delete=False) as tf:
                tf.write(rs.buf[: n * rs.stride].tobytes())
                path = tf.name
            try:
                p = subprocess.run([exe, path, str(K), str(M), str(cutoff), str(rs.read_len + 2)], capture_output=True, text=True, check=True, timeout=300)
                st = json.loads(p.stdout.strip().splitlines()[-1])
            finally:
                os.unlink(path)
            secs = st["process_read_s"] + st["prune_data_s"]
            shim = {"value": st["instances"] / secs, "unit": UNIT, "sample": f"first {n} reads, main's loop: process_read per read, then prune_data",
                    "process_read_s": st["process_read_s"], "prune_data_s": st["prune_data_s"], "walk_s": st["walk_s"], "kmers": st["kmers"],
                    "id_nodes": st["id_nodes"],
                    "note": "prune_data = H2D + GPU path + D2H + building the reference's pointer graph on one host core (one ZHashEntry per k-mer, "
                            "one ll_node per id); the graph build is what bounds this path"}
        except Exception as e:  # noqa: BLE001
            shim = {"value": None, "unavailable": f"{type(e).__name__}: {e}"}

    exchange_info = None
    if sharded is not None and stage_ms["exchange"] > 0:
        gbps = sharded.stats.sent_bytes_offrank / (stage_ms["exchange"] / 1e3) / 1e9
        exchange_info = {"GBps_per_dir_rank0": gbps, "nvlink_peak_GBps_per_dir": 900.0, "frac_of_nvlink": gbps / 900.0,
                         "bytes_sent_offrank_rank0": sharded.stats.sent_bytes_offrank, "ms_rank0": stage_ms["exchange"],
                         "note": "records this rank stored into the other owners' buffers (peer stores over NVLink, or NCCL all-to-all) divided by the "
                                 "time of the exchange stage on rank 0, which includes waiting for the slowest rank's scan"}
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "u64" if K <= 32 else "u128", "data": "synthetic",
            "config": config_dict(a, w, world), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu, "shim_path": shim, "table": stats, "input_split": input_split,
            "stage_ms_rank0": (dict(stage_ms, exchange_form=getattr(sharded, "exchange_kind", "nccl"),
                                    sent_bytes_offrank=sharded.stats.sent_bytes_offrank) if sharded is not None else None),
            "exchange": exchange_info, "table_digest": digest_info, "job_table": job, "selftest": selftest,
            "wall_s_timed_region": wall_s, "step_ms": step_ms,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    binner.close()


if __name__ == "__main__":
    main()
