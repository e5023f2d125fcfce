"""Read sets larger than one device, measured on one GPU: bench.py's config-3 read set (100 M x 150 bp, 12.0 G k-mer instances)
binned as P owner parts, one gbin_bin_reads_*_part call per part, in both forms (reads in pinned host memory; reads uploaded to
the device once).  The parts' digests must add up to config 3's pinned digest (profiles/expected_digests.json).

  python tools/parts_scale.py [--out DIR] [--skip-cfg3] [--reads N]

Prints one JSON line per measurement (and writes them to DIR/parts_scale.jsonl):
  * "memory": the context's device-memory high-water mark per k-mer instance of a one-part call at configs 2, 4, 5 and the
    config-3 shape (free memory before gbin_create minus free memory after the call; the context's buffers never shrink) —
    where gbin_plan_parts' bytes-per-instance constant comes from;
  * "cfg2_p1": config 2 as one part (host form) against gbin_bin_reads_host, alternated, wall time per call;
  * "cfg3": P from gbin_plan_parts and 2 P, both forms: per-part and total wall time, k-mers/s, bytes copied H2D / D2H, the
    high-water mark and the summed digest.
The card's name and power limit are read (nvidia-smi --query-gpu, read-only) in the same process."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
from genome_assembly_b200 import binding as B  # noqa: E402

CFG3_DIGEST = "98737683c4f9f64f"
OUT = []


def emit(d, out_dir):
    line = json.dumps(d)
    print(line, flush=True)
    OUT.append(line)
    if out_dir:
        with open(os.path.join(out_dir, "parts_scale.jsonl"), "a") as f:
            f.write(line + "\n")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement is still worth having; the line says the card was not read
        return f"unknown ({e})"


def free_bytes(torch):
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


def table_bytes(t):
    """Bytes of a table's arrays (what a host-form call copies to the host)."""
    return int(t.n_buckets) * 12 + 8 + int(t.n_kmers) * (8 * t.kmer_words + 8) + 8 + int(t.n_ids) * 4


def pinned_copy(lib, buf):
    p = lib.gbin_pinned_alloc(buf.nbytes)
    assert p, "gbin_pinned_alloc failed"
    dst = np.frombuffer((C.c_uint8 * buf.nbytes).from_address(p), dtype=np.uint8)
    dst[:] = buf
    return p, dst


def workload(name, reads=0):
    w = bench.workload_params(name, reads_override=reads, world=1)
    rs = bench.make_reads(w, 0, 1)
    return w, rs


def run_parts(torch, w, rs, P, form, d_reads=None, data_ptr=None, chunk_kb=0):
    """All P parts on a fresh context -> dict of timings, traffic, digest, high-water mark."""
    f0 = free_bytes(torch)
    b = B.Binner(w["k"], w["m"], w["cutoff"])
    if chunk_kb:
        b.set_tuning("part_chunk_kb", chunk_kb)
    if form == "host":
        rd = B.Binner._reads(data_ptr, rs.buf.nbytes, rs.n_reads, stride=rs.stride, read_len=rs.read_len)
    else:
        rd = B.Binner._reads(d_reads, d_reads.numel(), rs.n_reads, stride=rs.stride, read_len=rs.read_len)
    per_part, digests, inst, kmers, d2h, pipes = [], [], 0, 0, 0, []
    low = f0
    t_all = time.perf_counter()
    for p in range(P):
        t0 = time.perf_counter()
        t = b.bin_host_part_raw(rd, p, P) if form == "host" else b.bin_device_part_raw(rd, p, P)
        per_part.append(time.perf_counter() - t0)
        digests.append(b.table_digest(t))
        low = min(low, free_bytes(torch))
        inst += int(t.n_instances)
        kmers += int(t.n_kmers)
        d2h += table_bytes(t) if form == "host" else 0
        pipes.append(b.pipeline_info()["last_used"])
    total = time.perf_counter() - t_all
    b.close()
    return {"P": P, "form": form, "part_s": [round(x, 4) for x in per_part], "total_s": round(total, 4),
            "kmers_per_s": inst / sum(per_part), "instances": inst, "surviving_kmers": kmers,
            "h2d_bytes": rs.buf.nbytes * P if form == "host" else 0, "d2h_bytes": d2h, "pipelines": pipes,
            "high_water_bytes": f0 - low, "digest": "%016x" % (sum(digests) & ((1 << 64) - 1))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default="")
    ap.add_argument("--skip-cfg3", action="store_true")
    ap.add_argument("--reads", type=int, default=0, help="config-3 read count (default: all 100 M)")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "parts_scale.py measures on a GPU"
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    lib = B.load_library()
    emit({"card": card()}, a.out)

    # ---- high-water mark per instance of a one-part call (host form), the source of gbin_plan_parts' constant
    for name, reads in (("cfg2", 0), ("cfg4", 2_000_000), ("cfg5", 3_000_000), ("cfg3", 6_000_000)):
        w, rs = workload(name, reads)
        p, _view = pinned_copy(lib, rs.buf)
        r = run_parts(torch, w, rs, 1, "host", data_ptr=p)
        lib.gbin_pinned_free(p)
        emit({"memory": name, "reads": rs.n_reads, "read_len": rs.read_len, "K": w["k"], "M": w["m"], "instances": r["instances"],
              "high_water_bytes": r["high_water_bytes"], "bytes_per_instance": r["high_water_bytes"] / r["instances"],
              "reads_bytes": rs.buf.nbytes}, a.out)

    # ---- config 2 as one part against gbin_bin_reads_host, alternated on one context each
    w, rs = workload("cfg2")
    p, _view = pinned_copy(lib, rs.buf)
    rd = B.Binner._reads(p, rs.buf.nbytes, rs.n_reads, stride=rs.stride, read_len=rs.read_len)
    whole, part = B.Binner(w["k"], w["m"], w["cutoff"]), B.Binner(w["k"], w["m"], w["cutoff"])
    tw, tp = [], []
    for i in range(12):
        for b, acc, call in ((whole, tw, lambda b: b.bin_host_raw(rd)), (part, tp, lambda b: b.bin_host_part_raw(rd, 0, 1))):
            t0 = time.perf_counter()
            t = call(b)
            dt = time.perf_counter() - t0
            if i >= 2:  # the first two calls size the contexts' buffers and arenas
                acc.append(dt)
            dg = "%016x" % b.table_digest(t)
    emit({"cfg2_p1": True, "bin_reads_host_ms": [round(x * 1e3, 2) for x in tw], "host_part_ms": [round(x * 1e3, 2) for x in tp],
          "median_bin_reads_host_ms": statistics.median(tw) * 1e3, "median_host_part_ms": statistics.median(tp) * 1e3,
          "digest": dg}, a.out)
    whole.close()
    part.close()
    lib.gbin_pinned_free(p)

    if a.skip_cfg3:
        return
    # ---- config 3 on one GPU
    w, rs = workload("cfg3", a.reads)
    torch.cuda.empty_cache()
    p, _view = pinned_copy(lib, rs.buf)
    n_inst = rs.n_reads * (rs.read_len - w["k"] + 1)
    b = B.Binner(w["k"], w["m"], w["cutoff"])
    P = b.plan_parts(n_inst)
    b.close()
    emit({"cfg3_plan": True, "reads": rs.n_reads, "instances": n_inst, "free_bytes": free_bytes(torch), "P": P}, a.out)
    for PP in (P, 2 * P):
        r = run_parts(torch, w, rs, PP, "host", data_ptr=p)
        r.update(cfg3=True, reads=rs.n_reads, digest_ok=r["digest"] == CFG3_DIGEST or bool(a.reads))
        emit(r, a.out)
    d = torch.empty(rs.buf.nbytes, dtype=torch.uint8, device="cuda")
    d.copy_(torch.from_numpy(_view))
    del _view
    lib.gbin_pinned_free(p)
    b = B.Binner(w["k"], w["m"], w["cutoff"])
    Pd = b.plan_parts(n_inst)
    b.close()
    for PP in (Pd, 2 * Pd):
        r = run_parts(torch, w, rs, PP, "device", d_reads=d)
        r.update(cfg3=True, reads=rs.n_reads, digest_ok=r["digest"] == CFG3_DIGEST or bool(a.reads))
        emit(r, a.out)


if __name__ == "__main__":
    main()
