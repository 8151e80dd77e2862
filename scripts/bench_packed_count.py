"""Packed k-mer counting against ASCII counting on one GPU: hga_count_kmers on ASCII bases against hga_count_kmers_packed on the
case-folded 2-bit codes and exception runs, both from pinned host memory, at k = 19 and min_count = 2 (what jf_occurrences asks for per
file). The two arms alternate inside one call. The time of an arm is a host clock around the call, which copies the input, runs every
key-range pass and ends with a synchronise and the D2H of the result. Also reported: host-to-device bytes per call (from shapes), the
number of key-range passes (HGA_COUNT_STATS), the host packing rate of hga_host_pack_bases_folded, a digest of each arm's output (they
must be equal), and the card's name and power limit.

    python scripts/bench_packed_count.py [--configs 4] [--steps 2] [--warmup 1] [--exceptions]

One JSON line per config. The data come from bench.py's generators (same seeds). --exceptions injects N runs and lowercase stretches
into the reads before either arm sees them."""
import argparse
import ctypes as C
import hashlib
import json
import os
import re
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
from bench_packed_ingest import card, inject_exceptions  # noqa: E402

K, MIN_COUNT = 19, 2


class _KmerCounts(C.Structure):
    _fields_ = [("n", C.c_uint64), ("kmer", C.POINTER(C.c_uint64)), ("count", C.POINTER(C.c_uint32))]


def stderr_of(fn):
    """runs fn() with file descriptor 2 sent to a temporary file; returns (fn's result, what the library printed there)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        try:
            res = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        return res, f.read().decode(errors="replace")


def run(args, cfg, torch, np, hga_b200):
    c = bench.CONFIGS[cfg]
    dev = torch.device("cuda", 0)
    gsize = int(c["genome_mbp"] * 1e6)
    n_per_hap = max(1, int(c["coverage"] * gsize / c["mean_len"]))
    haps = bench.make_haplotypes(torch, dev, gsize, c["divergence"], args.seed, c["haplotypes"])
    lens, starts, flip, hap = bench.read_plan(torch, dev, gsize, n_per_hap, c["mean_len"], args.seed, c["len_sigma"], c["haplotypes"])
    n_reads = int(lens.shape[0])
    d_bases, d_off, n_bases = bench.synth_reads(torch, dev, list(haps), lens, starts, flip, hap, 0, n_reads, c["error"], args.seed, 0)
    del haps
    if args.exceptions:
        inject_exceptions(torch, d_bases, n_bases, args.seed + 1)
    torch.cuda.synchronize()

    # pinned host inputs (untimed): ASCII, and the folded codes + runs
    hb = torch.empty(n_bases + 64, dtype=torch.uint8, pin_memory=True)
    ho = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True)
    hb[:n_bases].copy_(d_bases[:n_bases]); ho.copy_(d_off)
    torch.cuda.synchronize()
    del d_bases, d_off
    torch.cuda.empty_cache()
    lib = hga_b200.load_library()
    n_bytes = (n_bases + 3) // 4
    hp = torch.empty(n_bytes + 64, dtype=torch.uint8, pin_memory=True)
    n_exc = C.c_uint64()
    exc_s = exc_e = None
    cap = 0
    for _ in range(2):
        t0 = time.perf_counter()
        rc = lib.hga_host_pack_bases_folded(C.c_void_p(hb.data_ptr()), n_bases, C.c_void_p(hp.data_ptr()),
                                            C.c_void_p(exc_s.data_ptr() if exc_s is not None else 0), C.c_void_p(exc_e.data_ptr() if exc_e is not None else 0),
                                            cap, C.byref(n_exc), 16)
        pack_s = time.perf_counter() - t0
        if rc == 0:
            break
        cap = int(n_exc.value)                                # too few run slots: retry with the exact count (the retry is timed)
        exc_s = torch.empty(max(cap, 1), dtype=torch.int64, pin_memory=True)
        exc_e = torch.empty(max(cap, 1), dtype=torch.int64, pin_memory=True)
    if rc != 0:
        raise hga_b200.HgaError(rc, lib.hga_last_error().decode())
    n_exc = int(n_exc.value)
    if exc_s is None:
        exc_s = torch.zeros(1, dtype=torch.int64, pin_memory=True); exc_e = torch.zeros(1, dtype=torch.int64, pin_memory=True)

    lib.hga_count_kmers.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.POINTER(_KmerCounts)]
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                           C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.argtypes = [C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.restype = None
    digests, n_kmers = {}, {}

    def call(arm):
        out = _KmerCounts()
        t0 = time.perf_counter()
        if arm == "ascii":
            rc = lib.hga_count_kmers(0, K, C.c_void_p(hb.data_ptr()), C.c_void_p(ho.data_ptr()), n_reads, MIN_COUNT, C.byref(out))
        else:
            rc = lib.hga_count_kmers_packed(0, K, C.c_void_p(hp.data_ptr()), 0, C.c_void_p(ho.data_ptr()), n_reads, C.c_void_p(exc_s.data_ptr()),
                                            C.c_void_p(exc_e.data_ptr()), n_exc, MIN_COUNT, C.byref(out))
        dt = time.perf_counter() - t0                         # the call ends with a synchronise and the D2H of the result
        if rc != 0:
            raise hga_b200.HgaError(rc, lib.hga_last_error().decode())
        dg = hashlib.sha256()
        if out.n:
            dg.update(np.ctypeslib.as_array(out.kmer, shape=(int(out.n),)).tobytes())
            dg.update(np.ctypeslib.as_array(out.count, shape=(int(out.n),)).tobytes())
        digests[arm] = dg.hexdigest()
        n_kmers[arm] = int(out.n)
        lib.hga_free_kmer_counts(C.byref(out))
        return dt

    arms = ("ascii", "packed")
    os.environ["HGA_COUNT_STATS"] = "1"
    passes = {}
    for _ in range(args.warmup):                              # warm-up of both arms; also reads the pass counts
        for arm in arms:
            _, err = stderr_of(lambda: call(arm))
            m = re.search(r"(\d+) key-range passes \((\d+) ranges split\)", err)
            passes[arm] = {"passes": int(m.group(1)), "splits": int(m.group(2))} if m else {"passes": 1, "splits": 0}
    del os.environ["HGA_COUNT_STATS"]
    ms = {a: [] for a in arms}
    for _ in range(args.steps):                                # alternating
        for arm in arms:
            ms[arm].append(call(arm) * 1e3)

    mean = lambda v: sum(v) / len(v)
    h2d_bytes = {"ascii": n_bases + (n_reads + 1) * 8, "packed": n_bytes + (n_reads + 1) * 8 + 16 * n_exc}
    line = {
        "config": cfg, "workload": c["name"], "k": K, "min_count": MIN_COUNT, "n_reads": n_reads, "n_bases": n_bases, "n_exc_runs": n_exc,
        "exceptions_injected": bool(args.exceptions), "steps": args.steps, "warmup": args.warmup,
        "count": {a: {"ms_per_call": mean(ms[a]), "ms_all": ms[a], "gbases_per_s": n_bases / (mean(ms[a]) * 1e-3) / 1e9, "h2d_bytes_per_call": h2d_bytes[a],
                      "key_range": passes.get(a)} for a in arms},
        "speedup_packed_over_ascii": mean(ms["ascii"]) / mean(ms["packed"]),
        "host_pack_folded_16_threads": {"gbases_per_s": n_bases / pack_s / 1e9, "s": pack_s},
        "n_kmers_out": n_kmers, "digest": digests, "digests_equal": digests["ascii"] == digests["packed"],
        "card": card(), "torch_device_name": torch.cuda.get_device_name(0),
    }
    print(json.dumps(line), flush=True)
    del hb, ho, hp
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[4], choices=sorted(bench.CONFIGS))
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=4000)
    ap.add_argument("--exceptions", action="store_true", help="inject N runs and lowercase stretches into the reads")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 1)
    import numpy as np
    import torch
    import hga_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_packed_count.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(0)
    bad = False
    for cfg in args.configs:
        bad |= not run(args, cfg, torch, np, hga_b200)["digests_equal"]
    if bad:
        raise SystemExit("bench_packed_count.py: the packed arm's k-mer counts differ from the ASCII arm's")


if __name__ == "__main__":
    main()
