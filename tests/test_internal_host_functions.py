"""CPU: the __host__ __device__ helpers of csrc/hga_internal.cuh compiled for the host (g++ against the CUDA headers, no GPU needed).

What the scan relies on without ever checking it at run time:
  * strand symmetry: the bit hash, the minimizer and with them the filter block / key bucket of a k-mer are the same for the k-mer and its reverse
    complement (the scan hashes whatever strand it reads; the table was built from canonical values);
  * the multi-GPU partition of the table slots (whole buckets round robin) is a bijection between slots and (owner, list number), and the inverse
    used by the index export (hga_capi.cu) is its inverse.
"""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hybrid-genome-assembler_b200", "csrc")
CUDA_INC = "/usr/local/cuda/include"

PROGRAM = r"""
#include "hga_internal.cuh"
#include <cstdio>
#include <random>
#include <set>
int main() {
    std::mt19937_64 rng(12345);
    long checked = 0;
    for (int k = 1; k <= 32; k++) {
        for (uint64_t n_kmers : {1000ull, 1000000ull, 40000000ull}) {
            const KmerGeom g = hga_make_geom(k, n_kmers);
            if (g.use_min && (g.m < 1 || g.m > 16 || g.W != k - g.m + 1 || g.W < 2 || g.W > HGA_MIN_W)) { printf("bad geometry k=%d m=%d W=%d\n", k, g.m, g.W); return 1; }
            for (int t = 0; t < 2000; t++) {
                uint64_t x = rng();
                if (k < 32) x &= (1ull << (2 * k)) - 1;
                const uint64_t r = hga_revcomp64(x, k);
                if (hga_revcomp64(r, k) != x) { printf("revcomp is not an involution k=%d\n", k); return 1; }
                const uint32_t hx = hga_bits_hash(x, g), hr = hga_bits_hash(r, g);
                if (hx != hr) { printf("bit hash not strand symmetric k=%d\n", k); return 1; }
                const uint32_t mx = hga_minimizer(x, hx, g), mr = hga_minimizer(r, hr, g);
                if (mx != mr) { printf("minimizer not strand symmetric k=%d m=%d\n", k, g.m); return 1; }
                if (hga_bits_mask(hx) == 0) { printf("empty filter mask\n"); return 1; }
                if (hga_start_sector(hx) >= HGA_BUCKET_SLOTS / HGA_SECTOR_SLOTS) { printf("sector out of range\n"); return 1; }
                checked++;
            }
        }
    }
    // slot partition: bijection slot <-> (owner, list), lists of one owner dense in [0, ceil(buckets / G) * 32)
    for (uint32_t G = 1; G <= 9; G++) {
        const uint32_t n_slots = 32 * 1237;
        std::set<uint64_t> seen;
        const uint32_t n_lists = (n_slots / 32 + G - 1) / G * 32;
        for (uint32_t s = 0; s < n_slots; s++) {
            const uint32_t o = hga_owner_of_slot(s, G), l = hga_list_of_slot(s, G);
            if (o >= G || l >= n_lists) { printf("owner / list out of range G=%u\n", G); return 1; }
            if (!seen.insert(((uint64_t) o << 32) | l).second) { printf("two slots share (owner, list) G=%u\n", G); return 1; }
            const uint32_t back = ((l / 32) * G + o) * 32 + l % 32;            // the inverse the index export uses
            if (back != s) { printf("inverse mapping wrong G=%u\n", G); return 1; }
            if (s % 32 && hga_owner_of_slot(s - 1, G) != o) { printf("a bucket is split between owners\n"); return 1; }
        }
    }
    printf("ok %ld\n", checked);
    return 0;
}
"""


@pytest.mark.skipif(not os.path.exists(os.path.join(CUDA_INC, "cuda_runtime.h")), reason="CUDA headers not installed")
def test_strand_symmetry_filter_mask_and_slot_partition(tmp_path):
    src, exe = str(tmp_path / "t.cpp"), str(tmp_path / "t")
    open(src, "w").write(PROGRAM)
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", CUDA_INC, "-I", CSRC, "-o", exe, src], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("ok "), r.stdout + r.stderr
