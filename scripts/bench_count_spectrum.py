"""One step of jf_occurrences' k sweep on one GPU: the distinct count of the reads at one k, as the sweep computed it before
(hga_count_kmers_packed with min_count = 1, every distinct k-mer copied to the host to read its number) against the spectrum
(hga_count_spectrum_packed with n_bins = 0, what the sweep calls now, and with n_bins = 10001). The input is bench.py's reads at a config,
packed case-folded as scripts/bench_packed_count.py packs them, in pinned host memory; k = 15, 17, 19. The three arms alternate inside
one call. The time of an arm is a host clock around the call, which copies the input, runs every key-range pass and ends with a
synchronise and the D2H of its result. Also reported per arm: n_distinct (equal across arms), the host bytes the arm materialises
(from shapes) and the key-range passes (HGA_COUNT_STATS), with the card's name and power limit.

    python scripts/bench_count_spectrum.py [--configs 2 4] [--ks 15 17 19] [--steps 1] [--warmup 1] [--out-dir profiles]

The old arm keeps about 36 B of host memory per distinct k-mer at its peak (the library's growing per-pass vectors, up to twice their
content at 12 B per k-mer, and the malloc'ed copy it returns). It is skipped, and the reason recorded, when that estimate from the
spectrum's n_distinct exceeds MemAvailable. Writes <out-dir>/count_spectrum_config<c>.jsonl (one line per k) and prints each line."""
import argparse
import ctypes as C
import json
import os
import re
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
from bench_packed_count import _KmerCounts, stderr_of  # noqa: E402
from bench_packed_ingest import card  # noqa: E402

SPECTRUM_BINS = 10001
OLD_PEAK_BYTES_PER_KMER = 36


class _KmerSpectrum(C.Structure):
    _fields_ = [("n_windows", C.c_uint64), ("n_distinct", C.c_uint64), ("max_count", C.c_uint64)]


def mem_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    raise RuntimeError("no MemAvailable in /proc/meminfo")


def packed_reads(args, cfg, torch, hga_b200):
    """bench.py's reads of config cfg, case-folded packed into pinned host memory: (packed, read_off, runs start, runs end, n_runs, n_reads, n_bases)"""
    c = bench.CONFIGS[cfg]
    dev = torch.device("cuda", 0)
    gsize = int(c["genome_mbp"] * 1e6)
    n_per_hap = max(1, int(c["coverage"] * gsize / c["mean_len"]))
    haps = bench.make_haplotypes(torch, dev, gsize, c["divergence"], args.seed, c["haplotypes"])
    lens, starts, flip, hap = bench.read_plan(torch, dev, gsize, n_per_hap, c["mean_len"], args.seed, c["len_sigma"], c["haplotypes"])
    n_reads = int(lens.shape[0])
    d_bases, d_off, n_bases = bench.synth_reads(torch, dev, list(haps), lens, starts, flip, hap, 0, n_reads, c["error"], args.seed, 0)
    del haps
    torch.cuda.synchronize()
    hb = torch.empty(n_bases + 64, dtype=torch.uint8, pin_memory=True)
    ho = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True)
    hb[:n_bases].copy_(d_bases[:n_bases]); ho.copy_(d_off)
    torch.cuda.synchronize()
    del d_bases, d_off
    torch.cuda.empty_cache()
    lib = hga_b200.load_library()
    hp = torch.empty((n_bases + 3) // 4 + 64, dtype=torch.uint8, pin_memory=True)
    n_exc = C.c_uint64()
    rc = lib.hga_host_pack_bases_folded(C.c_void_p(hb.data_ptr()), n_bases, C.c_void_p(hp.data_ptr()), None, None, 0, C.byref(n_exc), 16)
    cap = int(n_exc.value)
    exc_s = torch.zeros(max(cap, 1), dtype=torch.int64, pin_memory=True)
    exc_e = torch.zeros(max(cap, 1), dtype=torch.int64, pin_memory=True)
    if rc != 0:                                                # too few run slots: again with the exact count
        rc = lib.hga_host_pack_bases_folded(C.c_void_p(hb.data_ptr()), n_bases, C.c_void_p(hp.data_ptr()), C.c_void_p(exc_s.data_ptr()),
                                            C.c_void_p(exc_e.data_ptr()), cap, C.byref(n_exc), 16)
    if rc != 0:
        raise hga_b200.HgaError(rc, lib.hga_last_error().decode())
    del hb
    return hp, ho, exc_s, exc_e, int(n_exc.value), n_reads, n_bases


def run(args, cfg, torch, hga_b200):
    hp, ho, exc_s, exc_e, n_exc, n_reads, n_bases = packed_reads(args, cfg, torch, hga_b200)
    lib = hga_b200.load_library()
    lib.hga_count_kmers_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                           C.POINTER(_KmerCounts)]
    lib.hga_count_spectrum_packed.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32,
                                              C.c_void_p, C.POINTER(_KmerSpectrum)]
    lib.hga_free_kmer_counts.argtypes = [C.POINTER(_KmerCounts)]
    lib.hga_free_kmer_counts.restype = None
    inputs = (C.c_void_p(hp.data_ptr()), 0, C.c_void_p(ho.data_ptr()), n_reads, C.c_void_p(exc_s.data_ptr()), C.c_void_p(exc_e.data_ptr()), n_exc)
    hist = (C.c_uint64 * SPECTRUM_BINS)()
    lines = []
    for k in args.ks:
        distinct, maxc = {}, {}

        def call(arm):
            t0 = time.perf_counter()
            if arm == "count_min1":
                out = _KmerCounts()
                rc = lib.hga_count_kmers_packed(0, k, *inputs, 1, C.byref(out))
                dt = time.perf_counter() - t0                  # the call ends with a synchronise and the D2H of every distinct k-mer
                if rc == 0:
                    distinct[arm] = int(out.n)
                    lib.hga_free_kmer_counts(C.byref(out))
            else:
                sp = _KmerSpectrum()
                n_bins = 0 if arm == "spectrum_bins0" else SPECTRUM_BINS
                rc = lib.hga_count_spectrum_packed(0, k, *inputs, n_bins, hist if n_bins else None, C.byref(sp))
                dt = time.perf_counter() - t0                  # the call ends with the D2H of n_bins + 3 words
                distinct[arm], maxc[arm] = int(sp.n_distinct), int(sp.max_count)
            if rc != 0:
                raise hga_b200.HgaError(rc, lib.hga_last_error().decode())
            return dt

        arms = ["spectrum_bins0", "spectrum_bins10001", "count_min1"]
        os.environ["HGA_COUNT_STATS"] = "1"
        passes, skipped = {}, {}
        for _ in range(args.warmup):                           # warm-up of every arm; also reads the pass counts
            for arm in list(arms):
                if arm == "count_min1":
                    need, avail = OLD_PEAK_BYTES_PER_KMER * distinct["spectrum_bins0"], mem_available()
                    if need > avail:
                        skipped[arm] = (f"estimated host peak {need / 1e9:.1f} GB ({OLD_PEAK_BYTES_PER_KMER} B x {distinct['spectrum_bins0']} distinct k-mers) "
                                        f"exceeds MemAvailable {avail / 1e9:.1f} GB")
                        arms.remove(arm)
                        continue
                _, err = stderr_of(lambda: call(arm))
                m = re.search(r"(\d+) key-range passes \((\d+) ranges split\)", err)
                passes[arm] = {"passes": int(m.group(1)), "splits": int(m.group(2))} if m else {"passes": 1, "splits": 0}
        del os.environ["HGA_COUNT_STATS"]
        ms = {a: [] for a in arms}
        for _ in range(args.steps):                            # alternating
            for arm in arms:
                ms[arm].append(call(arm) * 1e3)
        mean = lambda v: sum(v) / len(v)
        host_bytes = {"spectrum_bins0": 3 * 8, "spectrum_bins10001": (SPECTRUM_BINS + 3) * 8 + SPECTRUM_BINS * 8}
        if "count_min1" in arms:
            host_bytes["count_min1"] = {"result": 12 * distinct["count_min1"], "peak_estimate": OLD_PEAK_BYTES_PER_KMER * distinct["count_min1"]}
        line = {
            "config": cfg, "workload": bench.CONFIGS[cfg]["name"], "k": k, "n_reads": n_reads, "n_bases": n_bases, "n_exc_runs": n_exc,
            "steps": args.steps, "warmup": args.warmup,
            "arms": {a: {"ms_per_call": mean(ms[a]), "ms_all": ms[a], "n_distinct": distinct[a], "host_bytes": host_bytes[a], "key_range": passes.get(a)} for a in arms},
            "skipped": skipped, "max_count": maxc, "n_distinct_equal": len({distinct[a] for a in arms}) == 1,
            "mem_available_bytes": mem_available(), "card": card(), "torch_device_name": torch.cuda.get_device_name(0),
        }
        if "count_min1" in arms:
            line["speedup_bins0_over_count_min1"] = mean(ms["count_min1"]) / mean(ms["spectrum_bins0"])
        print(json.dumps(line), flush=True)
        lines.append(line)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, f"count_spectrum_config{cfg}.jsonl"), "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")
    del hp, ho, exc_s, exc_e
    torch.cuda.empty_cache()
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4], choices=sorted(bench.CONFIGS))
    ap.add_argument("--ks", type=int, nargs="+", default=[15, 17, 19])
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=4000)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    args.warmup = max(args.warmup, 1)
    import torch
    import hga_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_count_spectrum.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(0)
    bad = False
    for cfg in args.configs:
        bad |= not all(line["n_distinct_equal"] for line in run(args, cfg, torch, hga_b200))
    if bad:
        raise SystemExit("bench_count_spectrum.py: the arms' distinct counts differ")


if __name__ == "__main__":
    main()
