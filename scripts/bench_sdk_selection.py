"""The SDK selection step of jf_occurrences on one GPU, after the counting input is loaded: the host path it replaced (every file
counted with hga_count_kmers_packed(min_count = 2) and copied to the host, hga_host_sdk_merge, hga_host_sdk_specificity,
hga_host_sdk_select on the whole merged table) against the device path (hga_sdk_count_packed over all files, hga_sdk_specificity,
hga_sdk_range, hga_host_sdk_select on the range). The input is bench.py's reads at a config, one file per haplotype (bench.py
generates the reads haplotype by haplotype), packed case-folded into pinned host memory as scripts/bench_count_spectrum.py packs them.
The two arms alternate inside one call. lower / upper come from the specificity table: the k-mers of the last threshold (100.01, the
ones in one file only) around the weighted median m of their totals, lower = max(2, m // 2), upper = 3 * m // 2; percent = 1.

    python scripts/bench_sdk_selection.py [--configs 2 4 5] [--k 19] [--steps 1] [--warmup 1] [--out-dir profiles]

Per arm: the host-clock time of each step (each call ends with a synchronise and its D2H), the host bytes the arm materialises (from
shapes), the merged n, and SHA-256 digests of the merged list, the table and the selected k-mers (equal across arms), with the card's
name and power limit read in the same call. The old arm holds about 12 B per per-file entry plus 20 B per entry of the merge output;
it is skipped, and the reason recorded, when 32 B x n_merged x n_files exceeds MemAvailable. Writes
<out-dir>/sdk_selection_config<c>.jsonl (one line per config) and prints it."""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
from bench_count_spectrum import mem_available, packed_reads  # noqa: E402
from bench_packed_ingest import card  # noqa: E402

THRESHOLDS = (70, 85, 90, 95, 99, 100, 100.01)
OLD_BYTES_PER_ENTRY = 32


def _digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _bounds(rows):
    t, o, u = rows
    m = t == THRESHOLDS[-1]
    occ, cnt = o[m].astype(np.int64), u[m].astype(np.int64)
    if not len(occ):
        return 2, 2
    med = int(occ[np.searchsorted(np.cumsum(cnt), cnt.sum() / 2)])
    return max(2, med // 2), 3 * med // 2


def run(args, cfg, torch, hga_b200):
    hp, ho, exc_s, exc_e, n_exc, n_reads, n_bases = packed_reads(args, cfg, torch, hga_b200)
    c = bench.CONFIGS[cfg]
    n_files = c["haplotypes"]
    n_per_hap = max(1, int(c["coverage"] * int(c["genome_mbp"] * 1e6) / c["mean_len"]))
    first = np.array([min(f * n_per_hap, n_reads) for f in range(n_files)] + [n_reads], dtype=np.uint64)
    off = ho.numpy().view(np.uint64)
    st = exc_s.numpy()[:n_exc].view(np.uint64); en = exc_e.numpy()[:n_exc].view(np.uint64)
    packed = np.frombuffer((C.c_uint8 * hp.numel()).from_address(hp.data_ptr()), dtype=np.uint8)
    k = args.k
    state = {}

    def old_arm():
        tm, t0 = {}, time.perf_counter()
        per_file = []
        for f in range(n_files):
            r0, r1 = int(first[f]), int(first[f + 1])
            b0, b1 = off[r0], off[r1]
            m = (en > b0) & (st < b1)
            es, ee = np.maximum(st[m], b0) - b0, np.minimum(en[m], b1) - b0
            per_file.append(hga_b200.capi.count_kmers_packed(packed, off[r0:r1 + 1] - b0, es, ee, k, min_count=2, first_base=int(b0)))
        tm["count_ms"] = (time.perf_counter() - t0) * 1e3; t0 = time.perf_counter()
        merged = hga_b200.capi.sdk_merge(per_file)
        tm["merge_ms"] = (time.perf_counter() - t0) * 1e3; t0 = time.perf_counter()
        rows = hga_b200.capi.sdk_specificity(merged[1], merged[2], THRESHOLDS)
        tm["table_ms"] = (time.perf_counter() - t0) * 1e3
        lo, hi = _bounds(rows)
        t0 = time.perf_counter()
        sel, n_sel, n_disc = hga_b200.capi.sdk_select(merged[1], merged[3], lo, hi, 1.0, 0)
        tm["select_ms"] = (time.perf_counter() - t0) * 1e3
        entries = sum(len(p[0]) for p in per_file)
        return tm, {"n_merged": len(merged[0]), "host_bytes": 12 * entries + 20 * (len(merged[0]) + 1) + len(merged[0]), "lower": lo, "upper": hi,
                    "n_selected": n_sel, "n_discriminative": n_disc, "digest_merged": _digest(*merged), "digest_table": _digest(*rows),
                    "digest_selection": _digest(merged[0][sel])}

    def new_arm(digest):
        tm, t0 = {}, time.perf_counter()
        t = hga_b200.capi.sdk_count_packed(packed, off, st, en, k, first, min_count=2)
        tm["count_merge_ms"] = (time.perf_counter() - t0) * 1e3; t0 = time.perf_counter()
        rows = t.specificity(THRESHOLDS)
        tm["table_ms"] = (time.perf_counter() - t0) * 1e3
        lo, hi = _bounds(rows)
        t0 = time.perf_counter()
        r = t.range(lo, hi)
        tm["range_ms"] = (time.perf_counter() - t0) * 1e3; t0 = time.perf_counter()
        sel, n_sel, n_disc = hga_b200.capi.sdk_select(r[1], r[3], lo, hi, 1.0, 0)
        tm["select_ms"] = (time.perf_counter() - t0) * 1e3
        info = {"n_merged": t.n, "host_bytes": 20 * len(r[0]) + len(r[0]) + 16 * len(rows[0]), "lower": lo, "upper": hi, "n_selected": n_sel,
                "n_discriminative": n_disc, "digest_table": _digest(*rows), "digest_selection": _digest(r[0][sel])}
        if digest:                                                   # the whole merged table, outside the timed steps
            info["digest_merged"] = _digest(*t.range())
        t.close()
        return tm, info

    arms, skipped, res = ["new", "old"], {}, {"new": [], "old": []}
    for _ in range(args.warmup):
        _, info = new_arm(True)
        state["new"] = info
        need, avail = OLD_BYTES_PER_ENTRY * info["n_merged"] * n_files, mem_available()
        if need > avail:
            skipped["old"] = f"estimated host bytes {need / 1e9:.1f} GB ({OLD_BYTES_PER_ENTRY} B x {info['n_merged']} merged k-mers x {n_files} files) exceed MemAvailable {avail / 1e9:.1f} GB"
            arms = ["new"]
        else:
            _, state["old"] = old_arm()
    for _ in range(args.steps):
        for arm in arms:
            res[arm].append(old_arm()[0] if arm == "old" else new_arm(False)[0])
    mean = lambda v: sum(v) / len(v)
    line = {"config": cfg, "workload": c["name"], "k": k, "n_files": n_files, "n_reads": n_reads, "n_bases": n_bases, "steps": args.steps, "warmup": args.warmup,
            "arms": {a: {"ms": {s: mean([r[s] for r in res[a]]) for s in res[a][0]}, "ms_all": res[a], **state[a]} for a in arms},
            "skipped": skipped, "mem_available_bytes": mem_available(), "card": card(), "torch_device_name": torch.cuda.get_device_name(0)}
    if "old" in arms:
        o, n = line["arms"]["old"], line["arms"]["new"]
        line["equal"] = all(o[key] == n[key] for key in ("n_merged", "digest_merged", "digest_table", "digest_selection", "lower", "upper"))
        line["total_ms"] = {a: sum(line["arms"][a]["ms"].values()) for a in arms}
    print(json.dumps(line), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, f"sdk_selection_config{cfg}.jsonl"), "w") as f:
        f.write(json.dumps(line) + "\n")
    del hp, ho, exc_s, exc_e, packed
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4, 5], choices=sorted(bench.CONFIGS))
    ap.add_argument("--k", type=int, default=19)
    ap.add_argument("--steps", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=4000)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    args.warmup = max(args.warmup, 1)
    import torch
    import hga_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench_sdk_selection.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(0)
    bad = [cfg for cfg in args.configs if run(args, cfg, torch, hga_b200).get("equal") is False]
    if bad:
        raise SystemExit(f"bench_sdk_selection.py: the arms differ at configs {bad}")


if __name__ == "__main__":
    main()
