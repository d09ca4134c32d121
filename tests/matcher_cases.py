"""Shapes, sample sheets and keys of the matcher path tests (test_gpu_matcher_paths.py, test_matcher_paths_host.py).

Every case names the pair of kernels frb_match must launch for it ("cand": match_idx1_cand_kernel + match_cand_kernel,
"sweep": match_idx1_kernel + match_kernel, "wide": match_idx1_wide_kernel + match_wide_kernel); the host test checks
those names against match_plan() of match_kernel.cuh, so that a changed threshold cannot quietly move a boundary case
onto another kernel."""
import random
import zlib

import numpy as np

SHAPE_ROWS = 48
# dual-index shapes (l1, l2) and the n of each that takes the candidate tables at SHAPE_ROWS rows
SHAPES = {
    "8+8": (8, 8, {0, 1, 2, 3}), "10+10": (10, 10, {0, 1, 2, 3}), "6+8": (6, 8, {0, 1, 2, 3}),
    "8+10": (8, 10, {0, 1, 2, 3}), "10+8": (10, 8, {0, 1, 2, 3}), "4+4": (4, 4, {0, 1, 2, 3}), "2+2": (2, 2, {0, 1}),
    "3+12": (3, 12, set()), "12+8": (12, 8, set()), "8+12": (8, 12, set()), "19+1": (19, 1, set()),
    "1+19": (1, 19, set()),
}


def n_values(l1, l2):
    """n = 0..4, n = the longer index (every row matches) and n = 25."""
    return sorted({0, 1, 2, 3, 4, max(l1, l2), 25})


# 10+10 sheets at the row counts where the choice changes: (n, rows, path, slots of each candidate table)
BOUNDARY = [
    (0, 1024, "cand", 2048), (0, 1025, "cand", 4096), (0, 2048, "cand", 4096), (0, 2049, "sweep", 0),
    (1, 512, "cand", 2048), (1, 513, "cand", 4096), (1, 1024, "cand", 4096), (1, 1025, "sweep", 0),
    (2, 341, "cand", 2048), (2, 342, "cand", 4096), (2, 682, "cand", 4096), (2, 683, "sweep", 0),
    (3, 256, "cand", 2048), (3, 257, "cand", 4096), (3, 512, "cand", 4096), (3, 513, "sweep", 0),
    (1, 1, "cand", 2048), (1, 5000, "sweep", 0),
]
MAX_ROWS = 5000
SINGLE_L1 = [1, 8, 10, 11, 21]
WIDE_SHAPES = {"21+20": (21, 20), "20+21": (20, 21), "12+8": (12, 8), "8+12": (8, 12), "10+10": (10, 10)}
# more unique keys than twice the grid of each kernel: (l1, l2, n, wide, path) at SHAPE_ROWS rows
SCALE = {"cand": (10, 10, 1, False, "cand"), "sweep": (12, 8, 1, False, "sweep"), "wide": (12, 12, 1, True, "wide")}
GRID_BLOCKS_PER_SM = 8   # the largest grid any matcher kernel takes: sm_count * 8 blocks of 256 threads
GRID_THREADS_PER_BLOCK = 256


def plan_cases():
    """(label, l1, l2, n, rows, wide, path, slots or None) of every case the GPU tests run."""
    out = []
    for name, (l1, l2, cand) in SHAPES.items():
        for n in n_values(l1, l2):
            out.append((f"shape {name} n={n}", l1, l2, n, SHAPE_ROWS, False, "cand" if n in cand else "sweep", None))
    for n, rows, path, slots in BOUNDARY:
        out.append((f"boundary n={n} rows={rows}", 10, 10, n, rows, False, path, slots))
    for l1 in SINGLE_L1:
        for n in (0, 1, 2, l1):
            out.append((f"single {l1} n={n}", l1, 0, n, SHAPE_ROWS, False, "sweep", None))
    for name, (l1, l2) in WIDE_SHAPES.items():
        for n in (0, 1, 3):
            out.append((f"wide {name} n={n}", l1, l2, n, SHAPE_ROWS, True, "wide", None))
    out.append(("wide rows=5000", 10, 10, 1, MAX_ROWS, True, "wide", None))
    for name, (l1, l2, n, wide, path) in SCALE.items():
        out.append((f"scale {name}", l1, l2, n, SHAPE_ROWS, wide, path, None))
    return out


def rng_for(label):
    return random.Random(zlib.crc32(label.encode()))


_RC = str.maketrans("ATGCNatgcn", "TACGNtacgn")


def revcomp(s):
    return s.translate(_RC)[::-1]


def word(rnd, length, alphabet="ACGT"):
    return "".join(rnd.choice(alphabet) for _ in range(length))


def make_sheet(rnd, l1, l2, rows, odd=True):
    """A sheet whose rows draw idx1 / idx2 from small pools, so that rows share index values; some rows repeat
    under the same and under another sample name.  odd: a few rows in lowercase, and a few holding a symbol outside
    ACGTN ('x', '-'), which no read symbol equals.  l2 == 0: a single-index sheet."""
    p1 = [word(rnd, l1) for _ in range(max(2, rows // 2))]
    p2 = [word(rnd, l2) for _ in range(max(2, rows // 3))] if l2 else None
    ids, i1, i2 = [], [], []
    for r in range(rows):
        if r >= 2 and rnd.random() < 0.08:             # the same row again, under its own or another name
            s = rnd.randrange(r)
            ids.append(ids[s] if rnd.random() < 0.5 else f"s{r}")
            i1.append(i1[s])
            i2.append(i2[s] if l2 else None)
            continue
        ids.append(f"s{r}" if r == 0 or rnd.random() < 0.9 else f"s{rnd.randrange(r)}")
        i1.append(rnd.choice(p1))
        i2.append(rnd.choice(p2) if l2 else None)
    if odd and rows >= 8:
        for r in rnd.sample(range(rows), max(2, rows // 16)):
            i1[r] = i1[r].lower()
            if l2 and rnd.random() < 0.5:
                i2[r] = i2[r].lower()
        for r in rnd.sample(range(rows), max(2, rows // 16)):
            which = 1 if not l2 or rnd.random() < 0.5 else 2
            w = list(i1[r] if which == 1 else i2[r])
            w[rnd.randrange(len(w))] = rnd.choice("x-")
            if which == 1:
                i1[r] = "".join(w)
            else:
                i2[r] = "".join(w)
    return {"id": ids, "idx1": i1, "idx2": i2 if l2 else None}


def subst(rnd, w, k, alphabet="ACGTN"):
    """w as a read would carry it (uppercase, ACGTN) with k symbols changed to another symbol."""
    out = [c if c in "ACGTN" else rnd.choice("ACGT") for c in w.upper()]
    for p in rnd.sample(range(len(out)), min(k, len(out))):
        out[p] = rnd.choice([c for c in alphabet if c != out[p]] or ["A"])
    return "".join(out)


def edge_keys(rnd, idx, n, extra):
    """{key: reads}: for every row, keys at exactly n and exactly n + 1 substitutions in idx1 and in idx2 (the other
    index either exact, reverse-complemented, or holding N); then `extra` more keys: both indexes off by up to n + 1,
    idx2 in both orientations, N-only substitutions, an idx1 match with an idx2 of nowhere, and random keys."""
    keys = {}
    single = idx["idx2"] is None
    l1 = len(idx["idx1"][0])
    l2 = 0 if single else len(idx["idx2"][0])
    rows = len(idx["id"])

    def put(a, b=None):
        keys.setdefault(a if single else a + "+" + b, rnd.randrange(1, 60))

    def other(r):
        b = idx["idx2"][r]
        return rnd.choice([subst(rnd, b, 0), subst(rnd, revcomp(b), 0), subst(rnd, b, 1, "N")])

    for r in range(rows):
        for k in (n, n + 1):
            if single:
                put(subst(rnd, idx["idx1"][r], k))
                continue
            put(subst(rnd, idx["idx1"][r], k), other(r))
            put(subst(rnd, idx["idx1"][r], rnd.choice([0, n])), subst(rnd, rnd.choice([idx["idx2"][r], revcomp(idx["idx2"][r])]), k))
    for _ in range(extra):
        r = rnd.randrange(rows)
        kind = rnd.randrange(5)
        a = subst(rnd, idx["idx1"][r], rnd.randrange(n + 2))
        if single:
            put(a if kind < 3 else word(rnd, l1, "ACGTN") if kind == 3 else subst(rnd, idx["idx1"][r], l1, "N"))
        elif kind == 0:
            put(a, subst(rnd, idx["idx2"][rnd.randrange(rows)], rnd.randrange(n + 2)))
        elif kind == 1:
            put(a, subst(rnd, revcomp(idx["idx2"][r]), rnd.randrange(n + 2)))
        elif kind == 2:
            put(subst(rnd, idx["idx1"][r], n, "N"), subst(rnd, idx["idx2"][r], n + 1, "N"))
        elif kind == 3:
            put(a, word(rnd, l2))                       # idx1 matches, idx2 most likely in neither orientation
        else:
            put(word(rnd, l1, "ACGTN"), word(rnd, l2, "ACGTN"))
    return keys


_CODES = np.frombuffer(b"ACGTN", np.uint8)


def scale_keys(seed, idx, n, count):
    """`count` unique dual-index keys (numpy-generated): 80 % an idx1 within n substitutions of a sheet row (idx2:
    that row's, its reverse complement, or random, up to n + 1 substitutions), 20 % random."""
    rng = np.random.default_rng(seed)
    l1, l2 = len(idx["idx1"][0]), len(idx["idx2"][0])
    up = lambda col: np.array([list(s.upper().encode()) for s in col], np.uint8)
    s1 = up(idx["idx1"])
    s2 = up(idx["idx2"])
    s2rc = up([revcomp(s) for s in idx["idx2"]])
    m = int(count * 2.5) + 64
    rows = rng.integers(0, len(idx["id"]), m)
    near = rng.random(m) < 0.8
    a = np.where(near[:, None], s1[rows], _CODES[rng.integers(0, 4, (m, l1))])
    pick = rng.integers(0, 3, m)
    b = np.where((pick == 0)[:, None], s2[rows], np.where((pick == 1)[:, None], s2rc[rows],
                                                          _CODES[rng.integers(0, 4, (m, l2))]))
    for arr, lim in ((a, n), (b, n + 1)):
        for _ in range(lim):
            hit = rng.random(m) < 0.5
            pos = rng.integers(0, arr.shape[1], m)
            arr[hit, pos[hit]] = _CODES[rng.integers(0, 5, int(hit.sum()))]
    plus = np.full((m, 1), ord("+"), np.uint8)
    txt = np.ascontiguousarray(np.concatenate([a, plus, b], axis=1)).view(f"S{l1 + 1 + l2}").ravel()
    keys = list(dict.fromkeys(t.decode() for t in txt.tolist()))[:count]
    assert len(keys) == count
    cnt = rng.integers(1, 40, len(keys))
    return dict(zip(keys, cnt.tolist()))


def random_keys(seed, l1, l2, count):
    """About `count` unique random l1+l2 keys over ACGTN (N rarer)."""
    rng = np.random.default_rng(seed)
    m = int(count * 1.02) + 64
    codes = _CODES[np.minimum(rng.integers(0, 17, (m, l1 + 1 + l2)) // 4, 4)]
    codes[:, l1] = ord("+")
    txt = np.ascontiguousarray(codes).view(f"S{l1 + 1 + l2}").ravel()
    return list(dict.fromkeys(t.decode() for t in txt.tolist()))[:count]


def idx1_hits(keys, sheet_idx1, n):
    """Keys whose idx1 is within n substitutions of some row's (numpy, case-insensitive): the matcher's work list."""
    l1 = len(sheet_idx1[0])
    a = np.frombuffer("".join(k[:l1] for k in keys).upper().encode(), np.uint8).reshape(-1, l1)
    s = np.frombuffer("".join(sheet_idx1).upper().encode(), np.uint8).reshape(-1, l1)
    hits = 0
    for c in range(0, len(a), 20000):
        hits += int(((a[c:c + 20000, None, :] != s[None, :, :]).sum(axis=2) <= n).any(axis=1).sum())
    return hits
