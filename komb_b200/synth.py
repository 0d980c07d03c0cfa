"""Deterministic synthetic workloads for the KOMB hot path (SURVEY.md section 8(d)).

Everything here is *input generation* (host side, numpy): alignment-hit sets,
SAM text renderings of them for the CPU reference, R-MAT / ramp edge lists.
None of it is on the measured path.

Workload names follow BASELINE.json `configs`:
  cfg1  tiny SAM pair (substitute for the absent example_data quickstart)
  cfg2  1 M unitigs, 5 M read pairs, ~20 M hits (the single-GPU bench workload)
  cfg3  R-MAT unitig graph (scale/edge count parameterised)
  cfg5  deep-core "ramp" graph (analytic coreness)
"""
from __future__ import annotations

import io
from dataclasses import dataclass

import numpy as np

# hits per mate for cfg2: uniform over this multiset (mean 2.0)
CFG2_HITS_PER_MATE = np.array([1, 1, 2, 2, 2, 3, 3], dtype=np.int64)


@dataclass
class HitSet:
    """Parsed alignment hits of one mate file: hit i says read `read_key[i]`
    aligned to unitig `unitig[i]`.  This is the integer form the reference
    reaches after tokenising SAM (src/graph.cpp:221-235)."""

    read_key: np.ndarray  # uint32[H]
    unitig: np.ndarray    # uint32[H]

    @property
    def n_hits(self) -> int:
        return int(self.read_key.shape[0])


def _powerlaw_unitigs(rng: np.random.Generator, count: int, n: int, alpha: float) -> np.ndarray:
    """Inverse-CDF sample of p(u) ~ (u+1)^-alpha on [0, n): u = floor(n * x^(1/(1-alpha)))."""
    x = rng.random(count)
    u = np.floor(n * np.power(x, 1.0 / (1.0 - alpha))).astype(np.int64)
    np.minimum(u, n - 1, out=u)
    return u.astype(np.uint32)


def scramble_ids(u: np.ndarray, n: int) -> np.ndarray:
    """Fixed bijection on [0, n): u -> (u * A + B) mod n with gcd(A, n) = 1.  Real unitig ids carry no
    degree order; the power-law generator's do (low id = hub), which would unbalance a range partition."""
    a = 2654435761
    while np.gcd(a, n) != 1:
        a += 2
    return ((u.astype(np.uint64) * np.uint64(a) + np.uint64(12345)) % np.uint64(n)).astype(np.uint32)


def metagenome_hits(n_unitigs: int, n_read_pairs: int, seed: int = 11, alpha: float = 0.5,
                    read_offset: int = 0, local_window: int = 0, scramble: bool = False) -> tuple[HitSet, HitSet]:
    """cfg2-style hit sets for the two mate files.

    Read pair r has k1 hits in mate file 1 and k2 in mate file 2, k uniform over
    CFG2_HITS_PER_MATE; unitigs follow a power law.  File order is read order.
    `read_offset` shifts read keys (used to give each rank its own read range).
    `local_window` > 0 draws all hits of one read pair from a window of that
    many unitigs around a power-law centre (models repeats landing nearby).
    """
    rng = np.random.Generator(np.random.PCG64(seed))
    mates = []
    centre = None
    if local_window > 0:
        centre = _powerlaw_unitigs(rng, n_read_pairs, n_unitigs, alpha).astype(np.int64)
    for _ in range(2):
        k = CFG2_HITS_PER_MATE[rng.integers(0, len(CFG2_HITS_PER_MATE), size=n_read_pairs)]
        reads = np.repeat(np.arange(n_read_pairs, dtype=np.int64), k)
        h = int(k.sum())
        if local_window > 0:
            off = rng.integers(0, local_window, size=h)
            unitig = ((centre[reads] + off) % n_unitigs).astype(np.uint32)
        else:
            unitig = _powerlaw_unitigs(rng, h, n_unitigs, alpha)
        if scramble:
            unitig = scramble_ids(unitig, n_unitigs)
        mates.append(HitSet((reads + read_offset).astype(np.uint32), unitig))
    return mates[0], mates[1]


def repeat_family_hits(n_unitigs: int = 200_000, family_size: int = 2000, overlap: int = 300, n_families: int = 3,
                       reads_per_family: int = 750, n_background: int = 100_000, seed: int = 21) -> tuple[HitSet, HitSet]:
    """Repeats under `bwa mem -a`: every read of a repeat family hits all of the family's unitigs, so one read emits
    C(family_size, 2) clique pairs (the defaults give 4 497 750 000 from the families: more than 2^32).

    Family f holds `family_size` unitigs, `overlap` of them shared with family f + 1; ids are scrambled over
    [0, n_unitigs).  Each family read lists its unitigs in its own shuffled order, split over the two mates with 200
    unitigs (a tenth of the family) in both.  The families' reads come first, then `n_background` cfg2-style read pairs
    (metagenome_hits).  Both mate files are in read order."""
    rng = np.random.Generator(np.random.PCG64(seed))
    step = family_size - overlap
    fams = [scramble_ids(np.arange(f * step, f * step + family_size, dtype=np.uint32), n_unitigs) for f in range(n_families)]
    both = family_size // 10
    split = (family_size + both) // 2
    rk = [[], []]
    ut = [[], []]
    r = 0
    for fam in fams:
        for _ in range(reads_per_family):
            order = rng.permutation(fam)
            for m, part in enumerate((order[:split], order[split - both:])):
                rk[m].append(np.full(part.shape[0], r, np.uint32))
                ut[m].append(part)
            r += 1
    b1, b2 = metagenome_hits(n_unitigs, n_background, seed=seed + 1, read_offset=r)
    return (HitSet(np.concatenate(rk[0] + [b1.read_key]), np.concatenate(ut[0] + [b1.unitig])),
            HitSet(np.concatenate(rk[1] + [b2.read_key]), np.concatenate(ut[1] + [b2.unitig])))


def render_sam(hits: HitSet, n_unitigs: int, mate: int, unmapped_every: int = 0,
               with_header: bool = True, qname_suffix: bool = True) -> bytes:
    """Render a hit set as SAM text the reference tokeniser accepts
    (src/graph.cpp:215-238: QNAME is field 0, RNAME field 2; '@' lines skipped;
    RNAME '*' skipped).  Unitig names are their decimal ids; QNAME is
    `read<r>/<mate>` so that the reference's key `substr(1, find('/'))`
    (graph.cpp:235) joins the two mates of a read.
    """
    out = io.BytesIO()
    if with_header:
        out.write(b"@HD\tVN:1.6\tSO:unsorted\n")
        sq = "".join(f"@SQ\tSN:{u}\tLN:500\n" for u in range(n_unitigs))
        out.write(sq.encode())
        out.write(b"@PG\tID:synth\tPN:komb_b200.synth\n")
    suffix = f"/{mate}" if qname_suffix else ""
    rk = hits.read_key.tolist()
    ut = hits.unitig.tolist()
    lines = []
    for i, (r, u) in enumerate(zip(rk, ut)):
        if unmapped_every and i % unmapped_every == unmapped_every - 1:
            lines.append(f"read{r}x{suffix}\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\tIIII\n")
        flag = 0 if (i == 0 or rk[i - 1] != r) else 256
        lines.append(f"read{r}{suffix}\t{flag}\t{u}\t{1 + (i % 400)}\t60\t4M\t*\t0\t0\tACGT\tIIII\n")
    out.write("".join(lines).encode())
    return out.getvalue()


def tiny_sam_pair(seed: int = 1, n_unitigs: int = 30, n_reads: int = 60, max_hits: int = 5,
                  unmapped_every: int = 7, qname_suffix: bool = True,
                  with_header: bool = True) -> tuple[bytes, bytes, HitSet, HitSet]:
    """cfg1 substitute: a small deterministic SAM pair with headers, unmapped
    records, 0..max_hits hits per mate and reads that map in one mate only."""
    rng = np.random.Generator(np.random.PCG64(seed))
    mates = []
    for _ in range(2):
        k = rng.integers(0, max_hits + 1, size=n_reads)
        reads = np.repeat(np.arange(n_reads, dtype=np.int64), k)
        unitig = _powerlaw_unitigs(rng, int(k.sum()), n_unitigs, 0.5)
        mates.append(HitSet(reads.astype(np.uint32), unitig))
    sam1 = render_sam(mates[0], n_unitigs, 1, unmapped_every, with_header, qname_suffix)
    sam2 = render_sam(mates[1], n_unitigs, 2, unmapped_every, with_header, qname_suffix)
    return sam1, sam2, mates[0], mates[1]


def write_fasta(path: str, n_unitigs: int) -> None:
    """A placeholder unitigs FASTA (komb2 -u): the reference opens and parses it
    (src/graph.cpp:446,565-589) but never uses the result."""
    with open(path, "w") as f:
        for u in range(n_unitigs):
            f.write(f">{u} LN:i:8\nACGTACGT\n")


# ---------------------------------------------------------------------------
# edge-list workloads (cfg3 / cfg5)
# ---------------------------------------------------------------------------

def _scramble32(x: np.ndarray) -> np.ndarray:
    """Fixed bijection on uint32 (xorshift-multiply rounds), so vertex-range
    partitions of R-MAT ids are load balanced."""
    x = x.astype(np.uint64)
    m = np.uint64(0xFFFFFFFF)
    x = (x ^ (x >> np.uint64(16))) & m
    x = (x * np.uint64(0x7FEB352D)) & m
    x = (x ^ (x >> np.uint64(15))) & m
    x = (x * np.uint64(0x846CA68B)) & m
    x = (x ^ (x >> np.uint64(16))) & m
    return x.astype(np.uint32)


def rmat_edges(scale: int, n_edges: int, n_vertices: int | None = None, seed: int = 42,
               abcd=(0.57, 0.19, 0.19, 0.05), scramble: bool = True) -> tuple[np.ndarray, np.ndarray]:
    """R-MAT edge list (with duplicates and loops, as generated): `n_edges`
    (u, v) draws over 2^scale ids, ids scrambled then folded `mod n_vertices`."""
    rng = np.random.Generator(np.random.PCG64(seed))
    a, b, c, _ = abcd
    u = np.zeros(n_edges, dtype=np.uint32)
    v = np.zeros(n_edges, dtype=np.uint32)
    for _ in range(scale):
        r = rng.random(n_edges, dtype=np.float32)
        ubit = (r >= a + b).astype(np.uint32)
        vbit = (((r >= a) & (r < a + b)) | (r >= a + b + c)).astype(np.uint32)
        u = (u << np.uint32(1)) | ubit
        v = (v << np.uint32(1)) | vbit
    if scramble:
        u = _scramble32(u)
        v = _scramble32(v)
    n = n_vertices or (1 << scale)
    return (u % np.uint32(n)).astype(np.uint32), (v % np.uint32(n)).astype(np.uint32)


def ramp_edges(levels: int, per_level: int) -> tuple[np.ndarray, np.ndarray]:
    """cfg5 planted ramp (SURVEY.md 8(d)): vertices r_0..r_{L-1}, L = levels *
    per_level, c(j) = 1 + j // per_level; r_j is adjacent to r_{j+1..j+c(j)}
    (clipped at L-1) and the last levels+1 vertices form a clique.
    Coreness levels 1..levels-(levels+1)/per_level are all non-empty and the
    clique has coreness `levels` (checked against the BZ oracle in tests), so
    peeling needs about `levels` dependent rounds."""
    L = levels * per_level
    us, vs = [], []
    j = np.arange(L, dtype=np.int64)
    c = 1 + j // per_level
    for d in range(1, levels + 1):
        sel = j[(c >= d) & (j + d < L)]
        us.append(sel)
        vs.append(sel + d)
    # closing clique on the last levels+1 vertices
    t = np.arange(L - (levels + 1), L, dtype=np.int64)
    iu, iv = np.triu_indices(levels + 1, k=1)
    us.append(t[iu])
    vs.append(t[iv])
    u = np.concatenate(us).astype(np.uint32)
    v = np.concatenate(vs).astype(np.uint32)
    return u, v
