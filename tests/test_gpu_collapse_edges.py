"""Edge tests of collapse's distance kernels (csrc/collapse.cu) against an exact numpy oracle.

dcb_umi_pairs: complete small spaces, barcodes repeated as collapse passes them (one per group), lists whose raw pair list
overflows its first allocation in both forms, low-complexity UMIs, a list whose runs of equal variants cross tiles,
UMIs of 0-2 and 18-19 symbols, the all-pairs sweep at k = 0 and 3 on 200 k UMIs and at tile-count boundaries, and a
host model of the deletion-neighbourhood form (entry list, copy skipping, two-deletion rule, part hash) that predicts
every part of a split search exactly.

dcb_lev_leq: every distance pinned exactly through two verdicts around it at the W dispatch boundaries, on both the
3-plane and the byte path; the threshold ties of collapse's fractions percentlevdist / 100 (the double product that
rounds below or above the integer); batch shapes and buffer reuse on one context.

The oracle is a textbook Levenshtein DP vectorised over pairs (collapse_oracle.levenshtein pins it); the CPU-only tests
check it and the constructed inputs.
"""
import ctypes
import functools
import itertools
import random

import numpy as np
import pytest

import collapse_oracle as CO
from decombinator_b200 import _lib

SYMDEL_MIN = 4096                                  # csrc/collapse.cu: deletion neighbourhoods from this many UMIs


def symdel_first_cap(n):                           # first allocation of the raw pair list, deletion neighbourhoods
    return max(1 << 22, 96 * n)


def allpairs_first_cap(n):                         # ... and all pairs
    return max(1 << 20, 8 * n)


# ---- the oracle ---------------------------------------------------------------------------------------------------
def lev_np(A, la, B, lb, band=None):
    """Levenshtein distance of every pair (A[t, :la[t]], B[t, :lb[t]]): the textbook DP, one row of the matrix per step,
    vectorised over the pairs.  band=b: only the cells with |i - j| <= b are computed and every value is capped at b + 1;
    a path of cost <= b never leaves that band, so the result is min(distance, b + 1)."""
    A, B = np.asarray(A), np.asarray(B)
    la, lb = np.asarray(la, dtype=np.int64), np.asarray(lb, dtype=np.int64)
    P = len(la)
    if P == 0:
        return np.zeros(0, dtype=np.int32)
    top = int(la.max())
    if band is None:
        W = B.shape[1]
        cols = np.arange(W + 1, dtype=np.int32)
        prev = np.broadcast_to(cols, (P, W + 1)).copy()
        out = lb.astype(np.int32)                                  # la == 0
        for i in range(1, top + 1):
            cur = np.empty_like(prev)
            cur[:, 0] = i
            np.minimum(prev[:, :-1] + (A[:, i - 1, None] != B), prev[:, 1:] + 1, out=cur[:, 1:])   # substitution, deletion
            prev = np.minimum.accumulate(cur - cols, axis=1) + cols                                  # insertions along the row
            m = la == i
            out[m] = prev[m, lb[m]]
        return out
    # the band of row i is held as wd rows of P values (offset o = j - i + b), so that every step works on contiguous rows
    b = int(band)
    cap, wd = b + 1, 2 * b + 1
    AT = np.ascontiguousarray(A[:, :top].T)
    BT = np.zeros((max(B.shape[1], top) + 2 * b + 2, P), dtype=B.dtype)
    BT[b + 1:b + 1 + B.shape[1]] = B.T                              # B[:, j - 1] sits at row b + j
    prev = np.empty((wd, P), dtype=np.int16)
    for o in range(wd):
        prev[o] = o - b if o >= b else cap                 # row 0: cell (0, j) = j
    out = np.minimum(lb, cap).astype(np.int32)
    o_end = lb - la + b                                            # where cell (la, lb) sits in its row of the band
    for i in range(1, top + 1):
        cur = prev + (AT[i - 1][None, :] != BT[i:i + wd])           # substitution: cell (i - 1, j - 1), same offset
        np.minimum(cur[:-1], prev[1:] + 1, out=cur[:-1])            # deletion: cell (i - 1, j), next offset
        if i <= b:
            cur[:b - i] = cap                                      # j < 0
            cur[b - i] = i                                         # j = 0
        for o in range(1, wd):                                     # insertion: cell (i, j - 1)
            np.minimum(cur[o], cur[o - 1] + 1, out=cur[o])
        np.minimum(cur, cap, out=cur)
        prev = cur
        m = np.nonzero(la == i)[0]
        if len(m):
            ok = (o_end[m] >= 0) & (o_end[m] < wd)
            out[m] = cap
            out[m[ok]] = prev[o_end[m[ok]], m[ok]]
    return out


def lev_chunked(A, la, B, lb, band=None, chunk=1 << 20):
    return np.concatenate([lev_np(A[s:s + chunk], la[s:s + chunk], B[s:s + chunk], lb[s:s + chunk], band)
                           for s in range(0, len(la), chunk)] or [np.zeros(0, dtype=np.int32)])


def decode(codes):
    """UMI codes -> (symbols (n, 19) uint8, lengths int64)."""
    codes = np.asarray(codes, dtype=np.uint64)
    sym = np.stack([((codes >> np.uint64(3 * t)) & np.uint64(7)).astype(np.uint8) for t in range(19)], axis=1)
    ln = (codes >> np.uint64(58)).astype(np.int64)
    sym[np.arange(19)[None, :] >= ln[:, None]] = 0
    return sym, ln


def encode(rows):
    """list of symbol sequences (ints 0..7) -> uint64 codes"""
    out = np.zeros(len(rows), dtype=np.uint64)
    for i, r in enumerate(rows):
        v = len(r) << 58
        for t, s in enumerate(r):
            v |= int(s) << (3 * t)
        out[i] = v
    return out


def near_values(vals, k):
    """Pairs u < v of DISTINCT codes within k edits -> (u, v, d)."""
    sym, ln = decode(vals)
    m = len(vals)
    u, v = np.triu_indices(m, 1)
    keep = np.abs(ln[u] - ln[v]) <= k
    u, v = u[keep], v[keep]
    d = lev_chunked(sym[u], ln[u], sym[v], ln[v], band=k)
    near = d <= k
    return u[near], v[near], d[near]


def expand(inv, u, v):
    """Distinct-value pairs (u, v) (u == v: a value with itself) -> sorted row << 32 | col keys over list indices."""
    order = np.argsort(inv, kind="stable")
    counts = np.bincount(inv, minlength=int(inv.max()) + 1 if len(inv) else 0)
    starts = np.concatenate([[0], np.cumsum(counts)[:-1]])
    cu, cv = counts[u], counts[v]
    per = cu * cv
    total = int(per.sum())
    if total == 0:
        return np.zeros(0, dtype=np.uint64)
    pid = np.repeat(np.arange(len(u)), per)
    local = np.arange(total) - np.repeat(np.cumsum(per) - per, per)
    a = order[starts[u[pid]] + local // cv[pid]]
    b = order[starts[v[pid]] + local % cv[pid]]
    keep = a != b
    a, b = a[keep], b[keep]
    lo, hi = np.minimum(a, b).astype(np.uint64), np.maximum(a, b).astype(np.uint64)
    return np.unique((lo << np.uint64(32)) | hi)


class Oracle:
    """Exact pair lists of one UMI list: distances are computed once per pair of DISTINCT values (band kmax), so a
    barcode repeated 3 000 times costs nothing."""

    def __init__(self, codes, kmax=2):
        self.codes = np.asarray(codes, dtype=np.uint64)
        self.vals, self.inv = np.unique(self.codes, return_inverse=True)
        self.inv = self.inv.reshape(-1)
        self.u, self.v, self.d = near_values(self.vals, kmax)
        self.kmax = kmax
        self._near_key = np.sort(self.u.astype(np.uint64) * np.uint64(len(self.vals)) + self.v.astype(np.uint64))
        self._near_d = self.d[np.argsort(self.u.astype(np.uint64) * np.uint64(len(self.vals)) + self.v.astype(np.uint64))]
        self._pairs = {}

    def pairs(self, k):
        assert k <= self.kmax
        if k not in self._pairs:
            m = len(self.vals)
            sel = self.d <= k
            u = np.concatenate([np.arange(m), self.u[sel]])
            v = np.concatenate([np.arange(m), self.v[sel]])
            self._pairs[k] = expand(self.inv, u, v)
        return self._pairs[k]

    def value_distance(self, vi, vj):
        """distance of distinct values vi, vj (arrays), capped at kmax + 1"""
        lo, hi = np.minimum(vi, vj).astype(np.uint64), np.maximum(vi, vj).astype(np.uint64)
        key = lo * np.uint64(len(self.vals)) + hi
        d = np.full(len(key), self.kmax + 1, dtype=np.int32)
        if len(self._near_key):
            pos = np.minimum(np.searchsorted(self._near_key, key), len(self._near_key) - 1)
            found = self._near_key[pos] == key
            d[found] = self._near_d[pos[found]]
        d[vi == vj] = 0
        return d


# ---- host model of the deletion-neighbourhood form ----------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def variant_plan(L, d):
    """The kept positions of every variant of an L-symbol UMI in the order dcb_umi_variants_kernel writes them: none,
    then for each p the variant without p followed by those without p and a later symbol."""
    plan = [tuple(range(L))]
    if d >= 1:
        for p in range(L):
            c1 = [x for x in range(L) if x != p]
            plan.append(tuple(c1))
            if d >= 2:
                for q in range(p, L - 1):
                    plan.append(tuple(c1[:q] + c1[q + 1:]))
    return plan


def entry_list(codes, d):
    """(variant key, UMI id) entries as the variants kernel writes them and a stable sort by the 64-bit key orders them."""
    sym, ln = decode(codes)
    keys, ids = [], []
    for L in np.unique(ln):
        idx = np.nonzero(ln == L)[0]
        plan = variant_plan(int(L), d)
        K = np.empty((len(idx), len(plan)), dtype=np.uint64)
        for t, kept in enumerate(plan):
            v = np.full(len(idx), np.uint64(len(kept)) << np.uint64(58), dtype=np.uint64)
            for s, pos in enumerate(kept):
                v |= sym[idx, pos].astype(np.uint64) << np.uint64(3 * s)
            K[:, t] = v
        keys.append(K.ravel())
        ids.append(np.repeat(idx, len(plan)))
    keys, ids = np.concatenate(keys), np.concatenate(ids)
    order = np.argsort(ids, kind="stable")               # UMI after UMI, each in its own variant order
    keys, ids = keys[order], ids[order]
    order = np.argsort(keys, kind="stable")
    return keys[order], ids[order]


def copies(keys, ids):
    """entries that repeat the listing in front of them (same variant, same UMI)"""
    c = np.zeros(len(keys), dtype=bool)
    c[1:] = (keys[1:] == keys[:-1]) & (ids[1:] == ids[:-1])
    return c


def share_one_deletion(sa, sb, L):
    """Do two L-symbol UMIs (symbol rows) share a variant with one deletion each?  By definition: all L x L pairs."""
    if L == 0:
        return np.zeros(len(sa), dtype=bool)
    va = np.stack([np.delete(sa[:, :L], p, axis=1) for p in range(L)], axis=1)     # (P, L, L - 1)
    vb = np.stack([np.delete(sb[:, :L], p, axis=1) for p in range(L)], axis=1)
    return (va[:, :, None, :] == vb[:, None, :, :]).all(axis=3).any(axis=(1, 2))


def part_of(keys, n_parts):
    return (((keys * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(40)) & np.uint64(0xFFFFFFFF)) % np.uint64(n_parts)


def model_emissions(oracle, k):
    """Every (pair key, variant key) the runs kernel emits: each pair of listed UMIs inside a run of equal variants
    within k edits, except from a two-deletion run when the two (equal-length) UMIs share a one-deletion variant."""
    codes = oracle.codes
    keys, ids = entry_list(codes, k)
    keep = ~copies(keys, ids)
    keys, ids = keys[keep], ids[keep]
    start = np.concatenate([[0], np.nonzero(keys[1:] != keys[:-1])[0] + 1])
    size = np.diff(np.concatenate([start, [len(keys)]]))
    E, F = [], []
    for r in np.unique(size[size >= 2]):
        st = start[size == r]
        e, f = np.triu_indices(int(r), 1)
        E.append((st[:, None] + e).ravel())
        F.append((st[:, None] + f).ravel())
    if not E:
        return np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=np.uint64)
    E, F = np.concatenate(E), np.concatenate(F)
    ia, ib, key = ids[E], ids[F], keys[E]
    assert np.all(ia != ib)
    vi, vj = oracle.inv[ia], oracle.inv[ib]
    hit = oracle.value_distance(vi, vj) <= k
    _, ln = decode(codes)
    cand = np.nonzero(hit & ((key >> np.uint64(58)).astype(np.int64) + 2 == ln[ia]) & (ln[ia] == ln[ib]))[0]
    if len(cand):
        sym, vln = decode(oracle.vals)
        pu, pinv = np.unique(np.stack([vi[cand], vj[cand]], axis=1), axis=0, return_inverse=True)
        shared = np.zeros(len(pu), dtype=bool)
        for L in np.unique(vln[pu[:, 0]]):
            sel = vln[pu[:, 0]] == L
            shared[sel] = share_one_deletion(sym[pu[sel, 0]], sym[pu[sel, 1]], int(L))
        hit[cand[shared[pinv.reshape(-1)]]] = False
    lo, hi = np.minimum(ia, ib).astype(np.uint64), np.maximum(ia, ib).astype(np.uint64)
    return ((lo << np.uint64(32)) | hi)[hit], key[hit]


# ---- the lists ----------------------------------------------------------------------------------------------------
def complete_space(alphabet_size, length, seed):
    rows = list(itertools.product(range(alphabet_size), repeat=length))
    random.Random(seed).shuffle(rows)
    return encode(rows)


BC = {c: i for i, c in enumerate("ACGTNSL")}


def set_barcode(n1, n2):
    """collapse's set_barcode on N1 / N2: N1 of 4-5 padded with S, N1 of 7-8 cut to 5 bases + L"""
    if len(n1) < 6:
        return n1 + "S" * (6 - len(n1)) + n2
    if len(n1) > 6:
        return n1[:5] + "L" + n2
    return n1 + n2


def barcode_family(rng, n_parents, children, allow_n):
    """Distinct barcodes: random N1 / N2 parents and children one or two edits away in N1 (so N1 changes length) or N2."""
    bases = "ACGTN" if allow_n else "ACGT"
    out = []
    for _ in range(n_parents):
        n1 = "".join(rng.choice("ACGT") for _ in range(rng.choice((4, 5, 6, 6, 6, 7, 8))))
        n2 = "".join(rng.choice("ACGT") for _ in range(6))
        out.append(set_barcode(n1, n2))
        for _ in range(children):
            a, b = list(n1), list(n2)
            for _ in range(rng.choice((1, 1, 2))):
                op = rng.randrange(4)
                if op == 0 and len(a) < 8:
                    a.insert(rng.randrange(len(a) + 1), rng.choice(bases))
                elif op == 1 and len(a) > 4:
                    del a[rng.randrange(len(a))]
                elif op == 2:
                    a[rng.randrange(len(a))] = rng.choice(bases)
                else:
                    b[rng.randrange(6)] = rng.choice(bases)
            out.append(set_barcode("".join(a), "".join(b)))
    return list(dict.fromkeys(out))


def repeated(rng, barcodes, counts):
    umis = [bc for bc, c in zip(barcodes, counts) for _ in range(c)]
    rng.shuffle(umis)                                  # interleaved
    return umis


@functools.lru_cache(maxsize=None)
def barcode_list():
    rng = random.Random(31)
    bcs = barcode_family(rng, 40, 4, allow_n=True)
    counts = [rng.choice((rng.randint(1, 300), rng.randint(1, 12), rng.randint(1, 3))) for _ in bcs]
    return _lib.encode_umis_fixed(repeated(rng, bcs, counts)), bcs, counts


@functools.lru_cache(maxsize=None)
def retry_list(big, n_total, seed):
    """One barcode `big` times among other barcodes that recur 1-300 times: n_total UMIs in all."""
    rng = random.Random(seed)
    bcs = barcode_family(rng, 60, 3, allow_n=seed % 2 == 1)
    counts = [big]
    while sum(counts) < n_total:
        counts.append(min(n_total - sum(counts), rng.randint(1, 300)))
    bcs = bcs[:len(counts)]
    assert len(bcs) == len(counts) and min(counts[1:]) >= 1
    return _lib.encode_umis_fixed(repeated(rng, bcs, counts)), counts


def edits1(s, alphabet):
    out = set()
    for p in range(len(s) + 1):
        for ch in alphabet:
            out.add(s[:p] + ch + s[p:])
        if p < len(s):
            out.add(s[:p] + s[p + 1:])
            for ch in alphabet:
                out.add(s[:p] + ch + s[p + 1:])
    return out


@functools.lru_cache(maxsize=None)
def low_complexity_list():
    rng = random.Random(41)
    seeds = ["A" * 12, "C" * 12, "G" * 12, "T" * 12, "AC" * 6, "CA" * 6, "AG" * 6, "GT" * 6, "TA" * 6, "AAAAAACCCCCC",
             "AAAAAAAAAAAC", "CCCCCCAAAAAA"]
    umis = []
    for s in seeds:
        one = sorted(edits1(s, "ACGT"))
        two = sorted(set().union(*(edits1(x, "ACGT") for x in one)))
        umis += [s, s] + one + rng.sample(two, 250)
    umis = [u for u in umis if u]
    rng.shuffle(umis)
    return _lib.encode_umis_fixed(umis)


@functools.lru_cache(maxsize=None)
def length_list():
    """UMIs of 0, 1, 2, 18 and 19 symbols (19: the top symbol beside the length field) among 12-mers, with neighbours."""
    rng = random.Random(51)
    al = "ACGTNSL"
    umis = ["", "", "A", "L", "S", "AC", "CA", "LL", "AL", "NS"] + ["".join(p) for p in itertools.product("ACL", repeat=2)]
    for L in (18, 19, 19, 12):
        for _ in range(12):
            s = "".join(rng.choice(al) for _ in range(L - 1)) + rng.choice("NSL")
            umis.append(s)
            for x in rng.sample(sorted(edits1(s, al)), 20):
                if len(x) <= 19:
                    umis.append(x)
                    y = rng.choice(sorted(edits1(x, al)))
                    if len(y) <= 19:
                        umis.append(y)
    umis += ["".join(rng.choice("ACGT") for _ in range(12)) for _ in range(200)]
    rng.shuffle(umis)
    return _lib.encode_umis_fixed(umis)


def run_geometry(codes, d=2):
    """(run start, run length) of every run of equal variants, and the tile boundaries a repeated listing straddles."""
    keys, ids = entry_list(codes, d)
    start = np.concatenate([[0], np.nonzero(keys[1:] != keys[:-1])[0] + 1])
    size = np.diff(np.concatenate([start, [len(keys)]]))
    b = np.arange(256, len(keys), 256)
    split = b[(keys[b - 1] == keys[b]) & (ids[b - 1] == ids[b])]
    return keys, start, size, split


def geometry_candidate(n_fill, seed):
    """Fillers of 9 and 10 symbols (their shorter variants all sort in front of A^10), then every 12-mer within two
    substitutions of A^12: the run of A^10 holds 1 056 entries, A^12 alone 66 copies of it."""
    rng = random.Random(seed)
    core = [""]
    for r in range(12):
        core += ["A" * r + c + "A" * (11 - r) for c in "CGT"]
    for r, s in itertools.combinations(range(12), 2):
        for c1 in "CGT":
            for c2 in "CGT":
                x = ["A"] * 12
                x[r], x[s] = c1, c2
                core.append("".join(x))
    core[0] = "A" * 12
    rng.shuffle(core)
    frng = random.Random(7)
    fill = ["".join(frng.choice("CGT") for _ in range(9 + (i % 2))) for i in range(n_fill)]
    return _lib.encode_umis_fixed(fill + core)


def geometry_ok(codes):
    keys, start, size, split = run_geometry(codes)
    a10 = np.uint64(10 << 58)
    r = np.nonzero(keys[start] == a10)[0]
    if len(r) != 1:
        return False
    s, n = int(start[r[0]]), int(size[r[0]])
    return s > 0 and s % 256 == 0 and n > 3 * 256 and bool(np.any((split > s) & (split < s + n)))


@functools.lru_cache(maxsize=None)
def geometry_list():
    """The first (filler count, shuffle) found by the model for which the A^10 run starts at a positive multiple of
    256, spans more than three tiles, and has a repeated listing of one UMI split across a tile boundary."""
    for n_fill in range(1, 600):
        codes = geometry_candidate(n_fill, 0)
        keys, start, size, _ = run_geometry(codes)
        if int(start[np.nonzero(keys[start] == np.uint64(10 << 58))[0][0]]) % 256:
            continue
        for seed in range(50):
            codes = geometry_candidate(n_fill, seed)
            if geometry_ok(codes):
                return codes
    raise AssertionError("no list found")


LISTS = {
    "acgt_6mers": lambda: complete_space(4, 6, 1),
    "two_letter_12mers": lambda: complete_space(2, 12, 2),
    "three_letter_7mers": lambda: complete_space(3, 7, 3),
    "repeated_barcodes": lambda: barcode_list()[0],
    "low_complexity": low_complexity_list,
    "run_geometry": geometry_list,
    "lengths_0_2_18_19": length_list,
}


# the lists whose split search is checked part by part against the model (in the repeated barcodes a run holds up to
# 300 listings of one barcode, which the model would pair up one by one)
MODEL_LISTS = sorted(set(LISTS) - {"repeated_barcodes"})


@functools.lru_cache(maxsize=None)
def oracle_of(name):
    return Oracle(LISTS[name](), 2)


@functools.lru_cache(maxsize=None)
def model_of(name, k):
    return model_emissions(oracle_of(name), k)


def model_share(name, k, part, n_parts):
    pairs, keys = model_of(name, k)
    return np.unique(pairs[part_of(keys, n_parts) == np.uint64(part)])


# ---- CPU: the oracle and the constructed inputs -------------------------------------------------------------------
def test_oracle_matches_collapse_oracle_on_random_pairs():
    rng = random.Random(3)
    A, B, la, lb, strs = np.zeros((600, 40), np.uint8), np.zeros((600, 45), np.uint8), [], [], []
    for t in range(600):
        al = rng.choice(("AC", "ACGT", "ACGTNSLX"))
        a = "".join(rng.choice(al) for _ in range(rng.randrange(0, 41)))
        b = list(a)
        for _ in range(rng.randrange(0, 16)):
            op = rng.randrange(3)
            if op == 0 and b:
                b[rng.randrange(len(b))] = rng.choice(al)
            elif op == 1 and b:
                del b[rng.randrange(len(b))]
            elif len(b) < 45:
                b.insert(rng.randrange(len(b) + 1), rng.choice(al))
        b = "".join(b)
        A[t, :len(a)] = [ord(c) for c in a]
        B[t, :len(b)] = [ord(c) for c in b]
        la.append(len(a)); lb.append(len(b)); strs.append((a, b))
    want = np.array([CO.levenshtein(a, b) for a, b in strs])
    assert np.array_equal(lev_np(A, la, B, lb), want)
    assert np.array_equal(lev_np(B, lb, A, la), want)
    for band in (0, 1, 2, 3, 5):
        assert np.array_equal(lev_np(A, la, B, lb, band), np.minimum(want, band + 1)), band
    assert (want > 5).sum() > 50 and (want <= 2).sum() > 50


@pytest.mark.parametrize("name", ["acgt_6mers", "two_letter_12mers", "three_letter_7mers"])
def test_oracle_matches_collapse_oracle_on_complete_spaces(name):
    codes = LISTS[name]()
    sym, ln = decode(codes)
    assert len(np.unique(codes)) == len(codes) == {"acgt_6mers": 4096, "two_letter_12mers": 4096, "three_letter_7mers": 2187}[name]
    rng = np.random.default_rng(5)
    i, j = rng.integers(0, len(codes), 2000), rng.integers(0, len(codes), 2000)
    s = ["".join("ACGTNSLX"[c] for c in sym[x, :ln[x]]) for x in range(len(codes))]
    want = np.array([CO.levenshtein(s[a], s[b]) for a, b in zip(i, j)])
    assert np.array_equal(lev_np(sym[i], ln[i], sym[j], ln[j], band=2), np.minimum(want, 3))
    o = oracle_of(name)
    near = {(int(a), int(b)) for a, b in zip(o.u, o.v)}
    vi, vj = np.searchsorted(o.vals, codes[i]), np.searchsorted(o.vals, codes[j])
    for a, b, w in zip(vi, vj, want):
        if a != b:
            assert ((min(a, b), max(a, b)) in near) == (w <= 2)


@pytest.mark.parametrize("name", MODEL_LISTS)
@pytest.mark.parametrize("k", [1, 2])
def test_model_of_deletion_neighbourhoods_equals_the_oracle(name, k):
    """The host model's emissions made unique are the oracle's pair list: every pair within k shares a run, and the
    two-deletion rule drops no pair that no one-deletion run emits."""
    pairs, _ = model_of(name, k)
    assert np.array_equal(np.unique(pairs), oracle_of(name).pairs(k))


def test_entry_list_model():
    """The model lists 1 + L (+ L (L - 1) / 2) variants per UMI, and a UMI listed twice under one variant (AAC minus
    either A) sits in neighbouring entries that the copy rule skips."""
    codes = encode([[0, 0, 1], [1, 0, 0], [0, 1, 0]])
    for d in (1, 2):
        keys, ids = entry_list(codes, d)
        assert len(keys) == 3 * (1 + 3 + (3 if d == 2 else 0))
        assert np.all(keys[1:] >= keys[:-1])
        ac = encode([[0, 1]])[0]
        e = np.nonzero((keys == ac) & (ids == 0))[0]
        assert len(e) == 2 and e[1] == e[0] + 1 and copies(keys, ids)[e[1]]
    keys, ids = entry_list(codes, 2)
    first_a = np.nonzero(keys == encode([[0]])[0])[0]
    assert list(ids[first_a]) == [0, 0, 1, 1, 2, 2]           # UMI order inside a run, each UMI's copies together


def test_run_geometry_list():
    """The list the run walk is tested on: a run of more than three tiles that starts at a multiple of 256, with one
    UMI's repeated listing split across a tile boundary inside it."""
    codes = geometry_list()
    keys, start, size, split = run_geometry(codes)
    r = np.nonzero(keys[start] == np.uint64(10 << 58))[0][0]
    s, n = int(start[r]), int(size[r])
    assert s > 0 and s % 256 == 0 and n > 768
    inside = split[(split > s) & (split < s + n)]
    assert len(inside) >= 1
    _, ids = entry_list(codes, 2)
    assert ids[inside[0] - 1] == ids[inside[0]]


def test_repeated_barcodes_are_shaped_like_collapse():
    codes, bcs, counts = barcode_list()
    assert all(len(b) == 12 for b in bcs) and max(counts) > 250 and min(counts) == 1
    assert any("S" in b for b in bcs) and any("L" in b for b in bcs) and any("N" in b for b in bcs)
    assert any(b[4:6] == "SS" for b in bcs) and any(b[4:6] != "SS" and b[5] == "S" for b in bcs)   # N1 of 4 and of 5
    _, ln = decode(codes)
    assert np.all(ln == 12) and len(codes) == sum(counts)
    assert not np.all(codes[:-1] <= codes[1:])                           # interleaved, not grouped


def test_retry_lists_overflow_the_first_allocation():
    """The raw list holds every distinct pair at least once; these lists have more distinct pairs than the first
    allocation of the form they are run through."""
    codes, counts = retry_list(3000, 5000, 61)
    n, c = len(codes), counts[0]
    assert 4800 <= n <= 5200 and c * (c - 1) // 2 == 4_498_500 > symdel_first_cap(n)
    assert len(oracle_of_retry(3000, 5000, 61).pairs(1)) > symdel_first_cap(n)
    codes, counts = retry_list(1500, 2000, 62)
    n, c = len(codes), counts[0]
    assert c * (c - 1) // 2 == 1_124_250 > allpairs_first_cap(n) == 1 << 20


@functools.lru_cache(maxsize=None)
def oracle_of_retry(big, n_total, seed):
    return Oracle(retry_list(big, n_total, seed)[0], 2)


# ---- GPU: dcb_umi_pairs ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dist():
    d = _lib.Dist(0)
    yield d
    d.close()


def pair_keys(row, col):
    assert np.all(row < col)
    k = (row.astype(np.uint64) << np.uint64(32)) | col.astype(np.uint64)
    assert np.all(k[1:] > k[:-1])                                        # sorted, unique
    return k


def check_both_forms(dist, monkeypatch, codes, k, want):
    for force, method in (("0", "deletion neighbourhoods"), ("1000000000", "all pairs")):
        monkeypatch.setenv("DCB_UMI_SYMDEL_MIN", force)
        got = pair_keys(*dist.umi_pairs(codes, k))
        assert dist.last_method() == (method if 1 <= k <= 2 else "all pairs")
        assert len(got) == len(want) and np.array_equal(got, want), (force, k, len(got), len(want))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LISTS))
@pytest.mark.parametrize("k", [1, 2])
def test_umi_pairs_edges(dist, monkeypatch, name, k):
    """Both forms equal the oracle; each part of the deletion-neighbourhood form split into 2, 3 and 8 parts is
    exactly what the host model deals to it (MODEL_LISTS), and the parts add up to the whole."""
    codes = LISTS[name]()
    want = oracle_of(name).pairs(k)
    assert len(want) > 0
    check_both_forms(dist, monkeypatch, codes, k, want)
    monkeypatch.setenv("DCB_UMI_SYMDEL_MIN", "0")
    for n_parts in (2, 3, 8):
        got = []
        for part in range(n_parts):
            share = pair_keys(*dist.umi_pairs(codes, k, part=part, n_parts=n_parts))
            if name in MODEL_LISTS:
                assert np.array_equal(share, model_share(name, k, part, n_parts)), (n_parts, part)
            got.append(share)
        assert np.array_equal(np.unique(np.concatenate(got)), want)


@pytest.mark.gpu
def test_umi_pairs_switch_over(dist, monkeypatch):
    """With the variable unset: all pairs at 4 095 UMIs, deletion neighbourhoods at 4 096."""
    monkeypatch.delenv("DCB_UMI_SYMDEL_MIN", raising=False)
    codes = LISTS["acgt_6mers"]()
    assert len(codes) == SYMDEL_MIN
    for k in (1, 2):
        want = oracle_of("acgt_6mers").pairs(k)
        got = pair_keys(*dist.umi_pairs(codes, k))
        assert dist.last_method() == "deletion neighbourhoods" and np.array_equal(got, want)
        got = pair_keys(*dist.umi_pairs(codes[:-1], k))
        assert dist.last_method() == "all pairs"
        assert np.array_equal(got, want[(want & np.uint64(0xFFFFFFFF)) != np.uint64(SYMDEL_MIN - 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("big,n_total,seed", [(3000, 5000, 61), (1500, 2000, 62)])
def test_umi_pairs_raw_list_overflow(dist, monkeypatch, big, n_total, seed):
    """One barcode repeated 3 000 times (4 498 500 distinct pairs against a first allocation of 2^22 for deletion
    neighbourhoods), and 1 500 times in 2 000 (1 124 250 against 2^20 for all pairs): the search sizes the list again
    and walks once more, in both forms and in every part."""
    codes, counts = retry_list(big, n_total, seed)
    o = oracle_of_retry(big, n_total, seed)
    c = counts[0]
    if big == 3000:
        assert c * (c - 1) // 2 > symdel_first_cap(len(codes))
    assert c * (c - 1) // 2 > allpairs_first_cap(len(codes))
    for k in (1, 2):
        want = o.pairs(k)
        check_both_forms(dist, monkeypatch, codes, k, want)
        monkeypatch.setenv("DCB_UMI_SYMDEL_MIN", "0")
        for n_parts in (2, 3, 8):
            got = [pair_keys(*dist.umi_pairs(codes, k, part=p, n_parts=n_parts)) for p in range(n_parts)]
            assert np.array_equal(np.unique(np.concatenate(got)), want)


@pytest.mark.gpu
def test_umi_pairs_rejects_twenty_symbols(dist):
    codes = np.array([20 << 58, 12 << 58], dtype=np.uint64)
    for force in ("0", "1000000000"):
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv("DCB_UMI_SYMDEL_MIN", force)
            with pytest.raises(_lib.DcbError, match="longer than 19"):
                dist.umi_pairs(codes, 1)
            with pytest.raises(_lib.DcbError, match="longer than 19"):
                dist.umi_pairs(codes, 2, part=1, n_parts=3)


def random_umis(rng, n, length, alphabet=4):
    sym = rng.integers(0, alphabet, size=(n, length), dtype=np.uint64)
    codes = np.full(n, length << 58, dtype=np.uint64)
    for t in range(length):
        codes |= sym[:, t] << np.uint64(3 * t)
    return codes


@pytest.mark.gpu
def test_umi_pairs_exact_duplicates_at_size(dist):
    """k = 0 on 200 k UMIs (all pairs: deletion neighbourhoods serve k = 1 and 2 only): the pairs are exactly the
    equal values, checked over the whole list by a group-by."""
    rng = np.random.default_rng(71)
    codes = random_umis(rng, 200_000, 12)
    src = rng.integers(0, 200_000, 4000)
    dst = rng.integers(0, 200_000, 4000)
    codes[dst] = codes[src]                              # planted duplicates, some chained
    codes[rng.integers(0, 200_000, 700)] = codes[5]      # one value 700 times
    vals, inv = np.unique(codes, return_inverse=True)
    want = expand(inv.reshape(-1), np.arange(len(vals)), np.arange(len(vals)))
    assert len(want) > 240_000
    got = pair_keys(*dist.umi_pairs(codes, 0))
    assert dist.last_method() == "all pairs"
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_umi_pairs_three_edits_at_size(dist):
    """k = 3 on 200 k random 16-symbol UMIs plus planted neighbours at distance 1-4: every reported pair is within three
    edits, the planted ones at <= 3 are reported and those at 4 are not, and 50 sampled rows are complete."""
    rng = np.random.default_rng(72)
    n = 200_000
    codes = random_umis(rng, n, 16)
    sym, ln = decode(codes)
    prng = random.Random(72)
    planted, src = [], []
    while len(planted) < 1200:
        i = prng.randrange(n)
        s = list(sym[i, :16])
        for _ in range(prng.randint(1, 4)):
            op = prng.randrange(3)
            if op == 0:
                s[prng.randrange(len(s))] = prng.randrange(4)
            elif op == 1 and len(s) > 12:
                del s[prng.randrange(len(s))]
            elif len(s) < 19:
                s.insert(prng.randrange(len(s) + 1), prng.randrange(4))
        planted.append(s); src.append(i)
    pc = encode(planted)
    ps, pl = decode(pc)
    src = np.array(src)
    pd = lev_np(sym[src], ln[src], ps, pl)
    keep = pd >= 1
    pc, src, pd = pc[keep], src[keep], pd[keep]
    assert all((pd == d).sum() > 100 for d in (1, 2, 3, 4))
    allc = np.concatenate([codes, pc])
    asym, aln = decode(allc)
    row, col = dist.umi_pairs(allc, 3)
    got = pair_keys(row, col)
    assert dist.last_method() == "all pairs"
    d = lev_chunked(asym[row], aln[row], asym[col], aln[col], band=3)
    assert np.all(d <= 3)
    tgt = (np.minimum(src, n + np.arange(len(src))).astype(np.uint64) << np.uint64(32)) | (n + np.arange(len(src))).astype(np.uint64)
    found = np.isin(tgt, got)
    assert np.all(found[pd <= 3]) and not np.any(found[pd == 4])
    for i in np.concatenate([rng.integers(0, n, 45), n + rng.integers(0, len(pc), 5)]):
        dd = lev_chunked(np.broadcast_to(asym[i], asym.shape), np.full(len(allc), aln[i]), asym, aln, band=3)
        want = set(np.nonzero(dd <= 3)[0].tolist()) - {int(i)}
        mine = set(col[row == i].tolist()) | set(row[col == i].tolist())
        assert mine == want, int(i)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [255, 256, 257, 512, 513, 768, 769, 1024, 1025])
def test_umi_pairs_all_pairs_at_tile_boundaries(dist, monkeypatch, n):
    """The upper triangle of tile pairs decoded from the block index, at 256 m and 256 m + 1 UMIs."""
    rng = np.random.default_rng(n)
    codes = random_umis(rng, n, 6)
    o = Oracle(codes, 3)
    monkeypatch.setenv("DCB_UMI_SYMDEL_MIN", "1000000000")
    for k in (0, 1, 2, 3):
        vals = o.d <= k
        want = expand(o.inv, np.concatenate([np.arange(len(o.vals)), o.u[vals]]), np.concatenate([np.arange(len(o.vals)), o.v[vals]]))
        got = pair_keys(*dist.umi_pairs(codes, k))
        assert np.array_equal(got, want), k
        if k >= 1 and n > 256:
            assert np.any((want >> np.uint64(32)) // np.uint64(256) != (want & np.uint64(0xFFFFFFFF)) // np.uint64(256))


@pytest.mark.gpu
def test_umi_pairs_context_reuse(monkeypatch):
    """Searches in a row on one context: each equals the oracle; 0 or 1 UMIs after a large search leave an empty list;
    an output smaller than the list is refused with DCB_ENOMEM."""
    d = _lib.Dist(0)
    try:
        monkeypatch.setenv("DCB_UMI_SYMDEL_MIN", "0")
        a, b = LISTS["low_complexity"](), LISTS["acgt_6mers"]()
        for codes, name in ((a, "low_complexity"), (b, "acgt_6mers"), (a, "low_complexity")):
            assert np.array_equal(pair_keys(*d.umi_pairs(codes, 2)), oracle_of(name).pairs(2))
        for small in (np.zeros(0, dtype=np.uint64), a[:1]):
            d.umi_pairs(b, 2)
            row, col = d.umi_pairs(small, 2)
            assert len(row) == 0 and len(col) == 0
        row, _ = d.umi_pairs(b, 1)
        L = _lib.lib()
        n = ctypes.c_uint64()
        keys = np.zeros(len(row), dtype=np.uint64)
        assert L.dcb_umi_pairs(d._h, None, 0, 0, keys.ctypes.data, len(row) - 1, ctypes.byref(n)) == -3   # DCB_ENOMEM
        assert n.value == len(row) and not keys.any()
        assert L.dcb_umi_pairs(d._h, None, 0, 0, keys.ctypes.data, len(row), ctypes.byref(n)) == 0
        assert np.array_equal(keys, oracle_of("acgt_6mers").pairs(1))
    finally:
        d.close()


# ---- dcb_lev_leq ------------------------------------------------------------------------------------------------
LA = (0, 1, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 511, 512)


def seq_pairs_oracle(seqs, a, b):
    """exact distance of every pair (seqs[a[t]], seqs[b[t]]), strings, through lev_np"""
    la = np.array([len(seqs[i]) for i in a])
    lb = np.array([len(seqs[i]) for i in b])
    W = max(1, int(max(la.max(initial=0), lb.max(initial=0))))
    A = np.zeros((len(a), W), np.int32)
    B = np.zeros((len(b), W), np.int32)
    for t, (i, j) in enumerate(zip(a, b)):
        A[t, :la[t]] = [ord(c) for c in seqs[i]]
        B[t, :lb[t]] = [ord(c) for c in seqs[j]]
    out = np.zeros(len(a), dtype=np.int32)
    order = np.argsort(la, kind="stable")                 # similar lengths together: fewer rows per chunk
    for s in range(0, len(a), 4096):
        idx = order[s:s + 4096]
        out[idx] = lev_np(A[idx], la[idx], B[idx], lb[idx])
    return out


def edited(rng, a, alphabet, n_edits, target_len):
    b = list(a)
    for _ in range(n_edits):
        op = rng.randrange(3)
        if op == 0 and b:
            b[rng.randrange(len(b))] = rng.choice(alphabet)
        elif op == 1 and b:
            del b[rng.randrange(len(b))]
        elif len(b) < 512:
            b.insert(rng.randrange(len(b) + 1), rng.choice(alphabet))
    while len(b) < target_len:
        b.insert(rng.randrange(len(b) + 1), rng.choice(alphabet))
    return "".join(b)


@functools.lru_cache(maxsize=None)
def distance_batch(path):
    """Pairs whose shorter side has a length of LA, the longer up to 512 symbols, 0-40 edits plus length differences,
    in both argument orders -> (seqs, a, b, la, d)."""
    rng = random.Random(81 if path == "planes" else 82)
    alphabet = "ACGTNSLX" if path == "planes" else "ACGTNacgt\xe9\xff\x80RY"
    seqs, a, b = [], [], []
    for la in LA:
        for t in range(28):
            x = "".join(rng.choice(alphabet) for _ in range(la))
            lb = la + (0 if t % 4 == 0 else rng.choice((1, 2, 5, 40, 512 - la)) if la < 512 else 0)
            y = edited(rng, x, alphabet, rng.randint(0, 40), max(la, min(lb, 512)))
            y = y[:512]
            if len(y) < la:
                continue
            seqs += [x, y]
            i = len(seqs) - 2
            a.append(i if t % 2 else i + 1)
            b.append(i + 1 if t % 2 else i)
    a, b = np.array(a, dtype=np.uint32), np.array(b, dtype=np.uint32)
    d = seq_pairs_oracle(seqs, a, b)
    la = np.array([min(len(seqs[i]), len(seqs[j])) for i, j in zip(a, b)])
    return seqs, a, b, la, d


def tie_cases():
    """(la, p, exact) for la <= 512, p = 1..100 with la * p divisible by 100: exact = la * p // 100, and how the
    double la * (p / 100) compares with it (-1 below, 0 equal, 1 above)."""
    out = []
    for la in range(1, 513):
        for p in range(1, 101):
            if la * p % 100 == 0:
                t = la * p // 100
                x = la * (p / 100)
                out.append((la, p, t, (x > t) - (x < t)))
    return out


@functools.lru_cache(maxsize=None)
def tie_batch(path):
    """For every tie case, pairs at distance exact - 1, exact and exact + 1 BY CONSTRUCTION: the shorter sequence has
    none of the symbol `z`, the other is it with s of its symbols replaced by z and i copies of z inserted, so the
    distance is s + i (each z costs an edit; s + i edits make it)."""
    rng = random.Random(91)
    alphabet, z = ("ACG", "T") if path == "planes" else ("ACGNRYKMS", "T")
    seqs, rows = [], []
    for la, p, t, rnd in tie_cases():
        for dd in (t - 1, t, t + 1):
            if dd < 0:
                continue
            ins_lo, ins_hi = max(0, dd - la), min(dd, 512 - la)
            if ins_lo > ins_hi:
                continue
            ins = rng.randint(ins_lo, ins_hi)
            x = [rng.choice(alphabet) for _ in range(la)]
            y = list(x)
            for pos in rng.sample(range(la), dd - ins):
                y[pos] = z
            for _ in range(ins):
                y.insert(rng.randrange(len(y) + 1), z)
            seqs += ["".join(x), "".join(y)]
            rows.append((len(seqs) - 2, len(seqs) - 1, la, p, dd, t, rnd))
    return seqs, rows


def test_tie_cases_round_both_ways():
    cases = tie_cases()
    assert sum(r < 0 for *_, r in cases) == 25 and sum(r > 0 for *_, r in cases) == 68
    assert (100, 29, 29, -1) in cases and (300, 21, 63, 0) in cases
    # a threshold taken in float decides some of these pairs otherwise than the double product does
    f32 = np.float32
    flips = sum((d <= la * (p / 100)) != (f32(d) <= f32(la) * f32(p / 100))
                for la, p, t, _ in cases for d in (t - 1, t, t + 1) if d >= 0)
    assert flips == 51


@pytest.mark.parametrize("path", ["planes", "bytes"])
def test_tie_pairs_have_their_distance(path):
    seqs, rows = tie_batch(path)
    assert len(rows) == 3 * len(tie_cases()) - 1            # all but distance 513 at 512 symbols
    rng = random.Random(5)
    sample = rng.sample(rows, 300) + [r for r in rows if r[2] <= 3 or r[2] >= 510][:200]
    d = seq_pairs_oracle(seqs, [r[0] for r in sample], [r[1] for r in sample])
    assert np.array_equal(d, [r[4] for r in sample])
    for i, j, la, p, dd, t, rnd in sample[:40]:
        if la <= 120:
            assert CO.levenshtein(seqs[i], seqs[j]) == dd
            assert CO.seqs_equivalent(seqs[i], seqs[j], p / 100) == (dd <= la * (p / 100))
    assert all(len(seqs[i]) == la <= len(seqs[j]) <= 512 for i, j, la, *_ in rows)


@pytest.mark.parametrize("path", ["planes", "bytes"])
def test_distance_batch_shapes(path):
    seqs, a, b, la, d = distance_batch(path)
    assert set(la.tolist()) == set(LA)
    assert np.any(d > 40) and np.any(d == 0) and len(set(d.tolist())) > 60
    sym, _, _ = _lib.encode_seqs(seqs)
    if path == "planes":
        assert sym.max() == 7
    else:
        assert sym.max() >= 0xE9 and len(set("".join(seqs))) >= 9
    assert any(len(seqs[i]) > len(seqs[j]) for i, j in zip(a, b)) and any(len(seqs[i]) < len(seqs[j]) for i, j in zip(a, b))
    rng = random.Random(1)
    for t in rng.sample(range(len(a)), 30):
        if len(seqs[a[t]]) * len(seqs[b[t]]) < 40_000:
            assert CO.levenshtein(seqs[a[t]], seqs[b[t]]) == d[t]


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["planes", "bytes"])
def test_lev_leq_pins_every_distance(dist, path):
    """For every pair at oracle distance d: true at frac (d + 0.5) / la, false at (d - 0.5) / la -- the GPU distance is
    d exactly.  One call per (la, d)."""
    seqs, a, b, la, d = distance_batch(path)
    sym, off, ln = _lib.encode_seqs(seqs)
    assert (sym.max() > 7) == (path == "bytes")
    groups = {}
    for t in range(len(a)):
        groups.setdefault((int(la[t]), int(d[t])), []).append(t)
    for (l, dd), ts in groups.items():
        ia, ib = a[ts], b[ts]
        if l == 0:
            for frac in (0.0, 0.5, 1.0):
                assert dist.lev_leq(sym, off, ln, ia, ib, frac).tolist() == [dd == 0] * len(ts)
            continue
        assert dist.lev_leq(sym, off, ln, ia, ib, (dd + 0.5) / l).all(), (l, dd)
        assert not dist.lev_leq(sym, off, ln, ia, ib, (dd - 0.5) / l).any(), (l, dd)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["planes", "bytes"])
def test_lev_leq_threshold_ties(dist, path):
    """Pairs at exactly len(shorter) * p / 100 - 1, + 0, + 1 edits at the fraction collapse passes (percentlevdist / 100):
    the verdict is the reference's double comparison, and the 25 products that round below the integer reject the pair
    at the exact distance."""
    seqs, rows = tie_batch(path)
    sym, off, ln = _lib.encode_seqs(seqs)
    assert (sym.max() > 7) == (path == "bytes")
    by_p = {}
    for r in rows:
        by_p.setdefault(r[3], []).append(r)
    below = 0
    for p, rs in sorted(by_p.items()):
        a = np.array([r[0] for r in rs], dtype=np.uint32)
        b = np.array([r[1] for r in rs], dtype=np.uint32)
        got = dist.lev_leq(sym, off, ln, b, a, p / 100)
        want = [dd <= la * (p / 100) for _, _, la, _, dd, _, _ in rs]
        assert got.tolist() == want, p
        for g, (_, _, la, _, dd, t, rnd) in zip(got, rs):
            if dd == t and rnd < 0:
                assert not g
                below += 1
    assert below == 25


@functools.lru_cache(maxsize=None)
def pool(seed, n, max_len):
    rng = random.Random(seed)
    base = ["".join(rng.choice("ACGTN") for _ in range(rng.randint(0, max_len))) for _ in range(n // 2)]
    return base + [edited(rng, x, "ACGT", rng.randint(0, 6), 0)[:max_len] for x in base]


@pytest.mark.gpu
def test_lev_leq_batch_shapes():
    """Pairs that name one sequence twice, pair counts off a multiple of 128, and large / small / large batches on one
    context (its device buffers are kept between calls): every verdict is the oracle's."""
    d = _lib.Dist(0)
    try:
        seqs = pool(101, 4000, 48)
        sym, off, ln = _lib.encode_seqs(seqs)
        same = np.arange(0, 4000, 7, dtype=np.uint32)
        assert d.lev_leq(sym, off, ln, same, same, 0.0).all()
        rng = np.random.default_rng(102)
        for n_pairs in (1, 127, 129, 255, 1000, 4097):
            a = rng.integers(0, 4000, n_pairs).astype(np.uint32)
            b = np.where(rng.random(n_pairs) < 0.5, (a + 2000) % 4000, rng.integers(0, 4000, n_pairs)).astype(np.uint32)
            dd = seq_pairs_oracle(seqs, a, b)
            mn = np.minimum(ln[a], ln[b])
            for frac in (0.1, 0.25):
                assert d.lev_leq(sym, off, ln, a, b, frac).tolist() == [x <= m * frac for x, m in zip(dd, mn)], (n_pairs, frac)
        for seed, n_seqs, max_len, n_pairs in ((103, 3000, 40, 50_000), (104, 20, 200, 3), (105, 2000, 48, 30_000),
                                               (106, 3000, 32, 80_000)):
            seqs = pool(seed, n_seqs, max_len)
            sym, off, ln = _lib.encode_seqs(seqs)
            prng = np.random.default_rng(seed)
            a = prng.integers(0, n_seqs, n_pairs).astype(np.uint32)
            b = np.where(prng.random(n_pairs) < 0.6, (a + n_seqs // 2) % n_seqs, prng.integers(0, n_seqs, n_pairs)).astype(np.uint32)
            dd = seq_pairs_oracle(seqs, a, b)
            mn = np.minimum(ln[a], ln[b])
            want = dd <= mn * 0.1
            assert n_pairs < 100 or (want.any() and not want.all())
            assert np.array_equal(d.lev_leq(sym, off, ln, a, b, 0.1), want), seed
    finally:
        d.close()
