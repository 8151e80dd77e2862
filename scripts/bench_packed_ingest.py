"""Packed 2-bit ingest against ASCII ingest on one GPU: the same end-to-end step as bench.py's `e2e` (scan from pinned host memory
through components, D2H of the components), once through hga_scan with ASCII bases and once through hga_scan_packed with 2-bit codes
and exception runs. The two arms alternate inside one call. Also reported: host-to-device bytes per step (from shapes), the scan stage
alone with its input already in HBM (hga_scan_device against hga_scan_packed_device), the host packing rate of hga_host_pack_bases at
1 and 16 threads, a digest of each arm's components (they must be equal), and the card's name and power limit.

    python scripts/bench_packed_ingest.py [--configs 4] [--steps 3] [--exceptions]

One JSON line per config. The data come from bench.py's generators (same seeds). --exceptions injects N runs and lowercase stretches
into the reads before either arm sees them, so that a workload with exception runs is measured as well."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:                                # the measurement stands without it; say so
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def inject_exceptions(torch, d_bases, n_bases, seed):
    """N runs (1 per 20 kbases, 1..500 bases) and lowercase stretches (1 per 20 kbases, 1..2000 bases), in place"""
    dev = d_bases.device
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    for kind, max_len in ((0, 500), (1, 2000)):
        m = max(1, n_bases // 20000)
        start = torch.randint(0, n_bases, (m,), device=dev, generator=g)
        length = torch.randint(1, max_len + 1, (m,), device=dev, generator=g)
        first = torch.cumsum(length, 0) - length
        total = int(length.sum())
        pos = torch.repeat_interleave(start, length, output_size=total) + torch.arange(total, device=dev) - \
            torch.repeat_interleave(first, length, output_size=total)
        pos = torch.clamp(pos, max=n_bases - 1)
        if kind == 0:
            d_bases[pos] = ord("N")
        else:
            v = d_bases[pos]
            d_bases[pos] = torch.where(v < 97, v + 32, v)


def run(args, cfg, torch, np, hga_b200):
    c = bench.CONFIGS[cfg]
    k = c["ks"][0]
    dev = torch.device("cuda", 0)
    gsize = int(c["genome_mbp"] * 1e6)
    n_per_hap = max(1, int(c["coverage"] * gsize / c["mean_len"]))
    haps = bench.make_haplotypes(torch, dev, gsize, c["divergence"], args.seed, c["haplotypes"])
    sdk = bench.discriminative_set(torch, haps, k)
    kmers = sdk.cpu().numpy().astype(np.uint64)
    del sdk
    lens, starts, flip, hap = bench.read_plan(torch, dev, gsize, n_per_hap, c["mean_len"], args.seed, c["len_sigma"], c["haplotypes"])
    n_reads = int(lens.shape[0])
    d_bases, d_off, n_bases = bench.synth_reads(torch, dev, list(haps), lens, starts, flip, hap, 0, n_reads, c["error"], args.seed, 0)
    del haps
    if args.exceptions:
        inject_exceptions(torch, d_bases, n_bases, args.seed + 1)
    torch.cuda.synchronize()

    # pinned host inputs (untimed): ASCII, and the packed codes + runs
    hb = torch.empty(n_bases + 64, dtype=torch.uint8, pin_memory=True)
    ho = torch.empty(n_reads + 1, dtype=torch.int64, pin_memory=True)
    hb[:n_bases].copy_(d_bases[:n_bases]); ho.copy_(d_off)
    torch.cuda.synchronize()
    lib = hga_b200.load_library()
    n_bytes = (n_bases + 3) // 4
    hp = torch.empty(n_bytes + 64, dtype=torch.uint8, pin_memory=True)
    n_exc = C.c_uint64()
    pack_rate = {}
    exc_s = exc_e = None
    for threads in (1, 16):
        cap = 0 if exc_s is None else exc_s.shape[0]
        for _ in range(2):
            t0 = time.perf_counter()
            rc = lib.hga_host_pack_bases(C.c_void_p(hb.data_ptr()), n_bases, C.c_void_p(hp.data_ptr()),
                                         C.c_void_p(exc_s.data_ptr() if exc_s is not None else 0), C.c_void_p(exc_e.data_ptr() if exc_e is not None else 0),
                                         cap, C.byref(n_exc), threads)
            dt = time.perf_counter() - t0
            if rc == 0:
                break
            cap = int(n_exc.value)                            # too few run slots: retry with the exact count (the retry is timed)
            exc_s = torch.empty(max(cap, 1), dtype=torch.int64, pin_memory=True)
            exc_e = torch.empty(max(cap, 1), dtype=torch.int64, pin_memory=True)
        if rc != 0:
            raise hga_b200.HgaError(rc, lib.hga_last_error().decode())
        pack_rate[f"threads_{threads}"] = {"gbases_per_s": n_bases / dt / 1e9, "s": dt}
    n_exc = int(n_exc.value)
    if exc_s is None:
        exc_s = torch.zeros(1, dtype=torch.int64, pin_memory=True); exc_e = torch.zeros(1, dtype=torch.int64, pin_memory=True)

    h = hga_b200.Handle(kmers, k, device=0)
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    digests = {}

    def step(arm):
        if arm == "ascii":
            h.scan_host_ptr(hb.data_ptr(), ho.data_ptr(), n_reads)
        else:
            h.scan_packed_host_ptr(hp.data_ptr(), 0, ho.data_ptr(), n_reads, exc_s.data_ptr(), exc_e.data_ptr(), n_exc)
        h.build_index()
        h.pair_count(min_score=1)
        h.select_edges(fraction=0.15)
        h.components(min_size=30)
        comp = h.get_components()                              # D2H: label per read + component list
        dg = hashlib.sha256()
        for key in ("label", "comp_label", "comp_size"):
            dg.update(comp[key].tobytes())
        digests[arm] = dg.hexdigest()

    def timed(fn):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    arms = ("ascii", "packed")
    for arm in arms:                                           # warm-up of both arms
        step(arm)
    e2e_ms = {a: [] for a in arms}
    h2d_ms = {a: [] for a in arms}
    for _ in range(args.steps):                                # alternating
        for arm in arms:
            e2e_ms[arm].append(timed(lambda: step(arm)))
            h2d_ms[arm].append(h.metrics()["h2d_ms"])
    metrics = h.metrics()

    # the scan stage alone with the input in HBM
    d_packed = torch.from_numpy(hp[:n_bytes].numpy()).to(dev)
    d_es = exc_s[:max(n_exc, 1)].to(dev); d_ee = exc_e[:max(n_exc, 1)].to(dev)
    torch.cuda.synchronize()
    scan_fn = {"ascii": lambda: h.scan_device(d_bases.data_ptr(), d_off.data_ptr(), n_reads, n_bases),
               "packed": lambda: h.scan_packed_device(d_packed.data_ptr(), 0, d_off.data_ptr(), n_reads, n_bases, d_es.data_ptr(), d_ee.data_ptr(), n_exc)}
    for arm in arms:
        scan_fn[arm]()
    scan_ms = {a: [] for a in arms}
    for _ in range(args.steps):
        for arm in arms:
            scan_ms[arm].append(timed(scan_fn[arm]))
    h.close()

    mean = lambda v: sum(v) / len(v)
    h2d_bytes = {"ascii": n_bases + (n_reads + 1) * 8, "packed": n_bytes + (n_reads + 1) * 8 + 16 * n_exc}
    line = {
        "config": cfg, "workload": c["name"], "k": k, "n_reads": n_reads, "n_bases": n_bases, "n_exc_runs": n_exc, "exceptions_injected": bool(args.exceptions),
        "steps": args.steps,
        "e2e": {a: {"gbases_per_s": n_bases / (mean(e2e_ms[a]) * 1e-3) / 1e9, "ms_per_step": mean(e2e_ms[a]), "ms_all": e2e_ms[a],
                    "h2d_ms_metric": mean(h2d_ms[a]), "h2d_bytes_per_step": h2d_bytes[a]} for a in arms},
        "scan_in_hbm": {a: {"ms": mean(scan_ms[a]), "ms_all": scan_ms[a], "gbases_per_s": n_bases / (mean(scan_ms[a]) * 1e-3) / 1e9} for a in arms},
        "host_pack": pack_rate,
        "components_digest": digests, "digests_equal": digests["ascii"] == digests["packed"],
        "n_components": int(metrics["n_components"]), "n_pairs": int(metrics["n_pairs"]),
        "card": card(), "torch_device_name": torch.cuda.get_device_name(0),
    }
    print(json.dumps(line), flush=True)
    del d_bases, d_off, d_packed, hb, ho, hp
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[4], choices=sorted(bench.CONFIGS))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=4000)
    ap.add_argument("--exceptions", action="store_true", help="inject N runs and lowercase stretches into the reads")
    args = ap.parse_args()
    import numpy as np
    import torch
    import hga_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_packed_ingest.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(0)
    bad = False
    for cfg in args.configs:
        bad |= not run(args, cfg, torch, np, hga_b200)["digests_equal"]
    if bad:
        raise SystemExit("bench_packed_ingest.py: the packed arm's components differ from the ASCII arm's")


if __name__ == "__main__":
    main()
