"""Index batches with chosen run layouts, the update's launch geometry, and exact expected tables for
the sparse SGD update tests (tests only).

The update (dlrm_jl_b200/csrc/update.cu) sorts each table's stream by row id and reduces it in tiles of
T entries, chunks of G tiles, and a fix-up for the runs that cross chunks.  Nearly all of its index logic
sits at run, tile and chunk boundaries, so these helpers build batches whose sorted stream has exactly
the run lengths a test asks for, restate the geometry that decides where the boundaries fall and which
fix-up path runs, and compute expected tables that are exact in any summation order."""
from dataclasses import dataclass
from typing import List

import numpy as np
import scipy.sparse

from oracle import oracle as O

INLINE_MAX_ENTRIES = 1 << 18     # kUpdateInlineMaxEntries (update.cu:41): larger batches use two launches
INLINE_SMEM_CHUNKS = 1024        # kInlineSmemChunks (update.cu:248): more chunks use the grouped fix-up


# ---- run layouts ---------------------------------------------------------------------------------
def lengths_from_ends(ends, L: int) -> np.ndarray:
    """Run lengths of a stream of L entries whose runs end (exclusively) at `ends`; the last run ends at L."""
    e = np.unique(np.asarray([x for x in ends if 0 < x < L], dtype=np.int64))
    return np.diff(np.concatenate([[0], e, [L]]))


def runs_to_indices(row_ids, lengths, B: int, rng) -> np.ndarray:
    """[B][P] indices whose row-sorted stream is row_ids[i] repeated lengths[i] times (row_ids ascending),
    in a seeded shuffle: the sorted stream, hence every run boundary, is fixed; the positions are not."""
    row_ids = np.asarray(row_ids, dtype=np.int64)
    lengths = np.asarray(lengths, dtype=np.int64)
    assert len(row_ids) == len(lengths) and np.all(lengths >= 1) and np.all(np.diff(row_ids) > 0)
    L = int(lengths.sum())
    assert L % B == 0, (L, B)
    return rng.permutation(np.repeat(row_ids, lengths)).reshape(B, L // B)


def chained_row_ids(nruns: List[int], rng) -> List[np.ndarray]:
    """Ascending row ids for each table's runs, with gaps (untouched rows in between), where table k's
    first run has the row id of table k-1's last run."""
    out, start = [], 0
    for n in nruns:
        gaps = rng.integers(1, 3, size=n)
        gaps[0] = 0
        ids = start + np.cumsum(gaps)
        out.append(ids)
        start = int(ids[-1])
    return out


def edge_ends(L: int, T: int, j: int) -> List[int]:
    """Runs ending next to every multiple c of T * 2^j: exclusive ends c - 1, c, c + 1 and c + 2 in turn, so
    the last entry of a run falls one before, on, one after or two after a tile / chunk edge."""
    step = T << j
    return [n * step + (-1, 0, 1, 2)[(n + j) % 4] for n in range(1, L // step + 1)]


def mixed_ends(L: int, chunk: int, lpr: int, nsub: int, rng, filler_runs: int = 500,
               ballot_rounds: int = 64) -> List[int]:
    """Run ends for a stream of L entries (chunk = G * T entries per CTA):
    three single entries; a run of exactly one chunk; a run that starts mid-chunk and spans more than
    nsub chunks (when it fits); then, alternating, runs longer than lpr chunks and runs that cross one
    chunk boundary (many heads in one table, mixed in each warp of the fix-up); random runs fill the rest."""
    ends, p = [], 0

    def put(e):
        nonlocal p
        if p < e < L:
            ends.append(e)
            p = e
            return True
        return False

    for _ in range(3):
        put(p + 1)
    c = -(-p // chunk) * chunk
    put(c)
    put(c + chunk)
    put(p + chunk // 2)
    if p + (nsub + 2) * chunk < L // 2:
        put(p + (nsub + 1) * chunk + 1)
    i = 0
    while i < ballot_rounds and p + (lpr + 5) * chunk < 3 * L // 4:
        put(p + (lpr + 1 + i % 3) * chunk)                  # p is mid-chunk: ends mid-chunk past the lpr-chunk window
        put(-(-p // chunk) * chunk + max(1, chunk // 4))    # crosses the next chunk boundary only
        put(p + 1)
        i += 1
    mean = max(2, (L - p) // filler_runs)
    while put(p + int(rng.integers(1, 2 * mean))):
        pass
    return ends


# ---- launch geometry -----------------------------------------------------------------------------
def _cdiv(a: int, b: int) -> int:
    return -(-a // b)


@dataclass
class UpdateGeom:
    vec: int          # floats per lane load: 4 if D % 4 == 0, else 1
    lpr: int          # lanes per row
    nch: int          # template NCH: 16-byte (or 4-byte) loads per lane, bucketed to 1, 2, 4, 8
    threads: int      # CTA size of the tiles kernel
    G: int            # lane groups (= tiles) per CTA
    tile: int         # entries per lane group
    chunks: List[int]  # CTAs per table
    inline: bool      # level 3 inside the tiles launch

    @property
    def chunk(self) -> int:
        return self.G * self.tile

    @property
    def nsub(self) -> int:
        return 256 // self.lpr

    def path(self, k: int) -> str:
        if not self.inline:
            return "two-launch"
        return "smem" if self.chunks[k] <= INLINE_SMEM_CHUNKS else "grouped"


def update_geom(D: int, Ls: List[int], tile_option: int = 0, sm_count: int = 148,
                two_launches: bool = False) -> UpdateGeom:
    """Restates launch_update_r / launch_update_t (update.cu:635-794):
    lanes_per_row_log2 (635-639), the NCH buckets (781-791), THREADS and G (675, 689),
    choose_update_tile from the total entry count (648-655, 691-695), tiles and chunks (708-709, 744-745)
    and the inline / two-launch switch (703-704)."""
    vec = 4 if D % 4 == 0 else 1
    C = D // vec
    l2 = 0
    while (1 << l2) < C and l2 < 5:
        l2 += 1
    lpr = 1 << l2
    n = _cdiv(C, lpr)
    nch = 1 if n == 1 else 2 if n == 2 else 4 if n <= 4 else 8
    threads = 128 if nch > 4 else 256
    G = threads // lpr
    total = int(sum(Ls))
    resident = threads * (3 if nch <= 1 else 2 if nch <= 2 else 1)
    capacity = sm_count * resident // lpr
    tile = min(32, max(4, _cdiv(_cdiv(total, capacity), 4) * 4))
    if 4 <= tile_option <= 32 and tile_option % 4 == 0:
        tile = tile_option
    chunks = [_cdiv(_cdiv(L, tile), G) for L in Ls]
    inline = total <= INLINE_MAX_ENTRIES and not two_launches
    return UpdateGeom(vec, lpr, nch, threads, G, tile, chunks, inline)


# ---- exact data ----------------------------------------------------------------------------------
# Table entries k / 32 with |k| <= 64 (exact in bf16), gradient entries k / 16 with |k| <= 7 and lr a power
# of two: every partial sum, lr * sum and x - lr * sum is exact in fp32 for any multiplicity below 2^20, so
# the expected table does not depend on the order in which the kernel adds.
def exact_tables(rows: List[int], D: int, rng) -> List[np.ndarray]:
    return [(rng.integers(-64, 65, size=(r, D)) / 32).astype(np.float32) for r in rows]


def exact_grads(B: int, D: int, rng) -> np.ndarray:
    return (rng.integers(-7, 8, size=(B, D)) / 16).astype(np.float32)


def row_sums(idx: np.ndarray, g: np.ndarray):
    """(uniq, counts, sums, abs_sums): for every distinct row of idx ([B][P]) the sum over its (b, p) of
    g[b] (and of |g[b]|) in float64."""
    B = g.shape[0]
    flat = np.asarray(idx).reshape(B, -1)
    P = flat.shape[1]
    uniq, inv, cnt = np.unique(flat.reshape(-1), return_inverse=True, return_counts=True)
    S = scipy.sparse.csr_matrix((np.ones(B * P), (inv.reshape(-1), np.repeat(np.arange(B), P))),
                                shape=(len(uniq), B))
    g64 = g.astype(np.float64)
    return uniq, cnt, S @ g64, S @ np.abs(g64)


def expected_exact(table: np.ndarray, idx: np.ndarray, g: np.ndarray, lr: float, bf16: bool = False) -> np.ndarray:
    """table[r] - lr * sum of g[b] over idx[b, p] = r, computed in float64; asserts that the result is
    representable in float32 (the exact-data premise), then rounds to bf16 for bf16-stored tables."""
    uniq, _cnt, acc, _ = row_sums(idx, g)
    new = table[uniq].astype(np.float64) - float(lr) * acc
    new32 = new.astype(np.float32)
    assert np.array_equal(new32.astype(np.float64), new), "test data must keep the update exact in fp32"
    out = table.copy()
    out[uniq] = O.to_bf16(new32) if bf16 else new32
    return out
