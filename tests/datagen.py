"""Seeded synthetic inputs for the categorization hot path (SURVEY.md §8d). Test/bench infrastructure.

Genome pair generation follows the reference's scripts/read_generator.py:158-162 (uniform ACGT; the second
haplotype is the first with per-base substitution probability `rate`, shift 1..3 mod 4). Read simulators
(art, nanosim-h, simlord) are not installed, so reads are drawn directly: uniform start, strand flip
p=0.5, substitution errors, constant quality.
"""
import os

import numpy as np

BASES = np.frombuffer(b"ACGT", dtype=np.uint8)
COMP = np.array([3, 2, 1, 0], dtype=np.uint8)


def random_genome(n, seed):
    return np.random.default_rng(seed).integers(0, 4, size=n, dtype=np.uint8)


def mutate(codes, rate, seed):
    rng = np.random.default_rng(seed)
    shift = (rng.random(codes.shape[0]) < rate).astype(np.uint8) * rng.integers(1, 4, size=codes.shape[0], dtype=np.uint8)
    return ((codes + shift) % 4).astype(np.uint8)


def to_ascii(codes):
    return BASES[codes].tobytes().decode()


def canonical_kmers(codes, k):
    """All canonical k-mer values of a code array (uint64), in window order (KmerIterator semantics)."""
    n = codes.shape[0] - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.uint64)
    fwd = np.zeros(n, dtype=np.uint64)
    rev = np.zeros(n, dtype=np.uint64)
    c = codes.astype(np.uint64)
    for j in range(k):
        fwd |= c[j:j + n] << np.uint64(2 * (k - 1 - j))
        rev |= (np.uint64(3) - c[j:j + n]) << np.uint64(2 * j)
    return np.minimum(fwd, rev)


def kmer_to_str(v, k):
    return "".join("ACGT"[(int(v) >> (2 * (k - 1 - i))) & 3] for i in range(k))


def discriminative_kmers(haplotypes, k, mode="exactly_one"):
    """Canonical k-mers present in exactly one haplotype (or absent from at least one: mode='not_all')."""
    sets = [np.unique(canonical_kmers(h, k)) for h in haplotypes]
    allk, counts = np.unique(np.concatenate(sets), return_counts=True)
    if mode == "exactly_one":
        return allk[counts == 1]
    return allk[counts < len(haplotypes)]


def sample_reads(codes, n_reads, length, seed, error_rate=0.0, length_sigma=0.0, min_len=1, max_len=None):
    """Returns a list of code arrays. length_sigma > 0 => lognormal lengths with that sigma around `length`."""
    rng = np.random.default_rng(seed)
    G = codes.shape[0]
    out = []
    for _ in range(n_reads):
        if length_sigma > 0:
            L = int(rng.lognormal(np.log(length) - 0.5 * length_sigma ** 2, length_sigma))
        else:
            L = length
        L = max(min_len, min(L, max_len or G, G))
        s = int(rng.integers(0, G - L + 1))
        r = codes[s:s + L].copy()
        if error_rate > 0:
            err = rng.random(L) < error_rate
            r[err] = (r[err] + rng.integers(1, 4, size=int(err.sum()), dtype=np.uint8)) % 4
        if rng.random() < 0.5:
            r = COMP[r[::-1]]
        out.append(r)
    return out


def write_fasta(path, reads, prefix="r", newline="\n"):
    with open(path, "w", newline="") as f:
        for i, r in enumerate(reads):
            s = r if isinstance(r, str) else to_ascii(r)
            f.write(f">{prefix}{i}{newline}{s}{newline}")


def write_fastq(path, reads, prefix="r", newline="\n"):
    with open(path, "w", newline="") as f:
        for i, r in enumerate(reads):
            s = r if isinstance(r, str) else to_ascii(r)
            f.write(f"@{prefix}{i}{newline}{s}{newline}+{newline}{'I' * len(s)}{newline}")


def write_kmers(path, values, k, newline="\n"):
    with open(path, "w", newline="") as f:
        for v in values:
            f.write(kmer_to_str(v, k) + newline)


def make_diploid_case(outdir, genome_size, divergence, k, read_len, coverage, seed, error_rate=0.0, fmt="fasta",
                      length_sigma=0.0, kmer_subsample=1.0):
    """Two haplotypes, one read file each, discriminative k-mer file. Returns (read_paths, kmer_path)."""
    os.makedirs(outdir, exist_ok=True)
    a = random_genome(genome_size, 1000 * seed)
    b = mutate(a, divergence, 1000 * seed + 1)
    paths = []
    for i, h in enumerate((a, b)):
        n_reads = max(1, int(coverage * genome_size / read_len))
        reads = sample_reads(h, n_reads, read_len, 1000 * seed + 10 + i, error_rate=error_rate, length_sigma=length_sigma,
                             min_len=min(50, genome_size))
        p = os.path.join(outdir, f"hap{i}.{ 'fq' if fmt == 'fastq' else 'fa'}")
        (write_fastq if fmt == "fastq" else write_fasta)(p, reads, prefix=f"h{i}_")
        paths.append(p)
    sdk = discriminative_kmers([a, b], k)
    if kmer_subsample < 1.0:
        rng = np.random.default_rng(1000 * seed + 99)
        sdk = sdk[rng.random(sdk.shape[0]) < kmer_subsample]
    # shuffle so that the file order is not the sorted order (ids must not depend on it)
    rng = np.random.default_rng(1000 * seed + 98)
    kp = os.path.join(outdir, f"{k}-mers.txt")
    write_kmers(kp, rng.permutation(sdk), k)
    return paths, kp


def make_polyploid_case(outdir, genome_size, divergence, k, read_len, coverage, seed, n_haplotypes=4, error_rate=0.0, length_sigma=0.0):
    """BASELINE config 5 in small: a base haplotype + independent mutated copies, one read file per haplotype, DENSE discriminative
    set = canonical k-mers absent from at least one haplotype. Returns (read_paths, kmer_path)."""
    os.makedirs(outdir, exist_ok=True)
    base = random_genome(genome_size, 1000 * seed)
    haps = [base] + [mutate(base, divergence, 1000 * seed + 1 + i) for i in range(n_haplotypes - 1)]
    paths = []
    for i, h in enumerate(haps):
        n_reads = max(1, int(coverage * genome_size / read_len))
        reads = sample_reads(h, n_reads, read_len, 1000 * seed + 10 + i, error_rate=error_rate, length_sigma=length_sigma, min_len=min(50, genome_size))
        p = os.path.join(outdir, f"hap{i}.fa")
        write_fasta(p, reads, prefix=f"h{i}_")
        paths.append(p)
    sdk = discriminative_kmers(haps, k, mode="not_all")
    rng = np.random.default_rng(1000 * seed + 98)
    kp = os.path.join(outdir, f"{k}-mers.txt")
    write_kmers(kp, rng.permutation(sdk), k)
    return paths, kp


def fuzz_case(seed):
    """Random small diploid case for the parity fuzz tests: (haplotypes, reads as code arrays, k, fraction, min_size, enrich_min)."""
    rng = np.random.default_rng(9000 + seed)
    k = int(rng.choice([11, 13, 15, 17, 19, 21, 25]))
    gsize = int(rng.integers(3000, 40000))
    div = float(rng.choice([0.01, 0.02, 0.03, 0.05]))
    long_reads = bool(rng.integers(0, 2))
    read_len = int(rng.integers(800, 4000)) if long_reads else int(rng.integers(80, 300))
    cov = float(rng.integers(8, 35))
    err = float(rng.choice([0.0, 0.005, 0.02, 0.06])) if long_reads else float(rng.choice([0.0, 0.005, 0.01]))
    a = random_genome(gsize, 9100 + seed)
    if rng.integers(0, 3) == 0:           # a repeat: k-mers that occur several times per read
        rep = a[:min(400, gsize // 4)].copy()
        pos = int(rng.integers(gsize // 2, gsize - rep.shape[0]))
        a[pos:pos + rep.shape[0]] = rep
    b = mutate(a, div, 9200 + seed)
    n = max(4, int(cov * gsize / read_len))
    reads = sample_reads(a, n, read_len, 9300 + seed, error_rate=err, length_sigma=0.5 if long_reads else 0.0, min_len=min(40, gsize)) + \
        sample_reads(b, n, read_len, 9400 + seed, error_rate=err, length_sigma=0.5 if long_reads else 0.0, min_len=min(40, gsize))
    order = rng.permutation(len(reads))   # haplotypes interleaved: read ids carry no haplotype information
    reads = [reads[i] for i in order]
    fraction = float(rng.choice([0.05, 0.15, 0.3, 0.6]))
    min_size = int(rng.choice([2, 3, 5, 10, 30]))
    enrich_min = int(rng.choice([1, 2, 5, 20, 40]))
    return [a, b], reads, k, fraction, min_size, enrich_min


def many_loci_case(n_loci, locus_len, reads_per_haplotype, read_len, seed, k=19, divergence=0.03, error_rate=0.005, repeat_every=0):
    """Many independent diploid loci sampled with short reads, read ids shuffled: (bases, read_off uint64, discriminative k-mers of
    every locus, sorted). Large selections and many scaffold components from one input. With repeat_every = r, every r-th locus has a
    tandem repeat (10 copies of a 40 bp unit) in one haplotype only: its k-mers occur several times per read, so a read with few hits
    can still share a high score with a read inside the repeat."""
    reads, kmers = [], []
    for i in range(n_loci):
        a = random_genome(locus_len, seed + 4 * i)
        b = mutate(a, divergence, seed + 4 * i + 1)
        if repeat_every and i % repeat_every == 0:
            at = locus_len // 2
            a = np.concatenate([a[:at], np.tile(random_genome(40, seed + 4 * i + 5), 10), a[at:]])
        reads += sample_reads(a, reads_per_haplotype, read_len, seed + 4 * i + 2, error_rate=error_rate) + \
            sample_reads(b, reads_per_haplotype, read_len, seed + 4 * i + 3, error_rate=error_rate)
        kmers.append(discriminative_kmers([a, b], k))
    seqs = [to_ascii(reads[i]).encode() for i in np.random.default_rng(seed).permutation(len(reads))]
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=off[1:])
    return b"".join(seqs), off, np.unique(np.concatenate(kmers))
