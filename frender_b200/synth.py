"""Deterministic synthetic FASTQ + sample sheets (SURVEY.md section 8d).

Every byte of read `g` depends only on (seed, g) through a counter-based hash, so
any chunking and any GPU count produce the same stream.  This numpy generator is
the slow host twin of the device generator in `csrc/frb_synth.cu`; the two are
checked byte-for-byte in `tests/test_gpu_synth.py`, which lets small host slices
stand in for the 400M-read device-generated lanes in parity tests.

Record layout (Illumina style, variable-length coordinates):
    @A00123:45:HXXXXXXXX:<lane>:<tile>:<x>:<y> <1|2>:N:0:<i7>[+<i5>]\n
    <read_len random ACGT>\n+\n<read_len x 'F'>\n
"""
from dataclasses import dataclass, field

import numpy as np

GOLD = np.uint64(0x9E3779B97F4A7C15)
M1 = np.uint64(0xBF58476D1CE4E5B9)
M2 = np.uint64(0x94D049BB133111EB)
DRAWS_PER_READ = 32          # stride of the draw counter per read
J_KIND, J_PARTNER, J_RAND7, J_RAND5, J_ERR0, J_COORD, J_SEQ1, J_SEQ2 = 0, 1, 2, 3, 4, 16, 17, 22
BASES = np.frombuffer(b"ACGT", dtype=np.uint8)
COMP = np.array([3, 2, 1, 0], dtype=np.uint8)      # A<->T, C<->G on 2-bit codes
PREFIX = b"@A00123:45:HXXXXXXXX:"


def mix64(z):
    z = np.asarray(z, dtype=np.uint64)
    z = (z ^ (z >> np.uint64(30))) * M1
    z = (z ^ (z >> np.uint64(27))) * M2
    return z ^ (z >> np.uint64(31))


def draw(seed, g, j):
    """j-th 64-bit draw of read ordinal(s) g."""
    g = np.asarray(g, dtype=np.uint64)
    ctr = g * np.uint64(DRAWS_PER_READ) + np.uint64(j + 1)
    return mix64(np.uint64(seed) + ctr * GOLD)


@dataclass
class SynthSpec:
    seed: int
    l1: int
    l2: int                                  # 0 => single index (no "+i5")
    ids: list
    sheet_i7: np.ndarray                     # [S, l1] 2-bit codes as supplied in the sheet
    sheet_i5: np.ndarray                     # [S, l2]
    emit_rc: np.ndarray                      # [S] bool: reads carry rc(i5) for this sample
    cdf: np.ndarray                          # [S] uint64 cumulative thresholds in 2^32 units
    lane: int = 1
    read_len: int = 151
    sub_t: int = 197                         # 0.3 % of 65536
    n_t: int = 66                            # 0.1 % of 65536
    rand_t: int = int(0.03 * 2 ** 32)
    hop_t: int = int(0.01 * 2 ** 32)
    combinatorial: tuple = field(default=None)

    @property
    def n_samples(self):
        return len(self.ids)

    def emit_i5(self):
        """[S, l2] codes actually written to reads (rc applied where flagged)."""
        out = self.sheet_i5.copy()
        flip = COMP[self.sheet_i5[:, ::-1]]
        out[self.emit_rc] = flip[self.emit_rc]
        return out

    def indexes(self):
        """The sheet as the reference's get_indexes would return it."""
        d = {"id": list(self.ids), "idx1": [codes_to_str(r) for r in self.sheet_i7]}
        d["idx2"] = [codes_to_str(r) for r in self.sheet_i5] if self.l2 else None
        return d

    def sheet_csv(self):
        """Illumina-style sheet text ([Header]..[Data] preamble, no blank lines)."""
        lines = ["[Header]", "IEMFileVersion,4", "Workflow,GenerateFASTQ", "[Reads]",
                 str(self.read_len), "[Data]"]
        if self.l2:
            lines.append("Sample_ID,Sample_Name,index,index2")
            for sid, a, b in zip(self.ids, self.sheet_i7, self.sheet_i5):
                lines.append(f"{sid},{sid},{codes_to_str(a)},{codes_to_str(b)}")
        else:
            lines.append("Sample_ID,Sample_Name,index")
            for sid, a in zip(self.ids, self.sheet_i7):
                lines.append(f"{sid},{sid},{codes_to_str(a)}")
        return "\n".join(lines) + "\n"


def codes_to_str(codes):
    return BASES[np.asarray(codes, dtype=np.uint8)].tobytes().decode()


def _index_set(rng, count, length, min_dist=3):
    """`count` index sequences of `length` with pairwise Hamming >= min_dist."""
    chosen = np.empty((0, length), dtype=np.uint8)
    while len(chosen) < count:
        cand = rng.integers(0, 4, size=(4 * count, length), dtype=np.uint8)
        for c in cand:
            if len(chosen) == 0 or ((chosen != c).sum(axis=1) >= min_dist).all():
                chosen = np.vstack([chosen, c[None]])
                if len(chosen) == count:
                    break
    return chosen


def make_spec(config, seed=1234, n_samples=None, lane=1, read_len=151):
    """Spec for one of BASELINE.json's configs ("C1".."C5", SURVEY.md 8d)."""
    shapes = {
        "C1": dict(l1=8, l2=8, s=96, hop=0.01, rc=True),
        "C2": dict(l1=10, l2=10, s=384, hop=0.01, rc=True),
        "C3": dict(l1=8, l2=8, s=384, hop=0.05, rc=False, grid=(24, 16)),
        "C4": dict(l1=10, l2=10, s=384, hop=0.01, rc=True),
        "C5": dict(l1=6, l2=0, s=96, hop=0.0, rc=False),
    }
    sh = shapes[config]
    s = n_samples or sh["s"]
    rng = np.random.default_rng(seed + int(config[1]))
    if "grid" in sh and s == sh["s"]:
        a, b = sh["grid"]
        set7, set5 = _index_set(rng, a, sh["l1"]), _index_set(rng, b, sh["l2"])
        i7 = np.repeat(set7, b, axis=0)
        i5 = np.tile(set5, (a, 1))
    else:
        i7 = _index_set(rng, s, sh["l1"], 3 if sh["l1"] > 6 else 2)
        i5 = _index_set(rng, s, sh["l2"]) if sh["l2"] else np.zeros((s, 0), np.uint8)
    w = rng.lognormal(0.0, 1.0, size=s)
    cum = np.floor(np.cumsum(w) / w.sum() * 2.0 ** 32).astype(np.uint64)
    cum[-1] = np.uint64(2 ** 32)
    emit_rc = (rng.random(s) < 0.5) if (sh["rc"] and sh["l2"]) else np.zeros(s, bool)
    return SynthSpec(seed=seed + int(config[1]), l1=sh["l1"], l2=sh["l2"],
                     ids=[f"S{n + 1:03d}" for n in range(s)], sheet_i7=i7, sheet_i5=i5,
                     emit_rc=emit_rc, cdf=cum, lane=lane, read_len=read_len,
                     hop_t=int(sh["hop"] * 2 ** 32), combinatorial=sh.get("grid"))


def index_codes(spec, g):
    """([N, l1], [N, l2]) symbol codes 0..3 = ACGT, 4 = N for reads g."""
    g = np.asarray(g, dtype=np.uint64)
    n = len(g)
    w0 = draw(spec.seed, g, J_KIND)
    sample = np.minimum(np.searchsorted(spec.cdf, w0 & np.uint64(0xFFFFFFFF), side="right"),
                        spec.n_samples - 1)
    kind = w0 >> np.uint64(32)
    is_rand = kind < np.uint64(spec.rand_t)
    is_hop = (~is_rand) & (kind < np.uint64(spec.rand_t + spec.hop_t))
    w1 = draw(spec.seed, g, J_PARTNER)
    partner = np.minimum(np.searchsorted(spec.cdf, w1 & np.uint64(0xFFFFFFFF), side="right"),
                         spec.n_samples - 1)
    i7 = spec.sheet_i7[sample].copy()
    emit5 = spec.emit_i5()
    i5 = emit5[np.where(is_hop, partner, sample)].copy() if spec.l2 else np.zeros((n, 0), np.uint8)
    r7, r5 = draw(spec.seed, g, J_RAND7), draw(spec.seed, g, J_RAND5)
    for p in range(spec.l1):
        i7[is_rand, p] = ((r7 >> np.uint64(2 * p)) & np.uint64(3)).astype(np.uint8)[is_rand]
    for p in range(spec.l2):
        i5[is_rand, p] = ((r5 >> np.uint64(2 * p)) & np.uint64(3)).astype(np.uint8)[is_rand]
    both = np.concatenate([i7, i5], axis=1)
    for p in range(spec.l1 + spec.l2):
        word = draw(spec.seed, g, J_ERR0 + p // 2) >> np.uint64(32 * (p % 2))
        e16 = (word & np.uint64(0xFFFF)).astype(np.int64)
        s16 = ((word >> np.uint64(16)) & np.uint64(0xFFFF)).astype(np.int64)
        sub = e16 < spec.sub_t
        isn = (~sub) & (e16 < spec.sub_t + spec.n_t)
        col = both[:, p].astype(np.int64)
        col = np.where(sub, (col + 1 + s16 % 3) % 4, col)
        col = np.where(isn, 4, col)
        both[:, p] = col.astype(np.uint8)
    return both[:, :spec.l1], both[:, spec.l1:]


SYMS = np.frombuffer(b"ACGTN", dtype=np.uint8)


def keys_of(spec, g0, g1):
    """Index strings ("i7+i5" or "i7") of reads g0..g1-1, without building FASTQ."""
    a, b = index_codes(spec, np.arange(g0, g1, dtype=np.uint64))
    out = []
    for x, y in zip(SYMS[a], SYMS[b]):
        out.append(x.tobytes().decode() + ("+" + y.tobytes().decode() if spec.l2 else ""))
    return out


def generate(spec, g0, g1, read_no=1, index_read=None):
    """FASTQ bytes of reads g0..g1-1 of mate `read_no` (1 or 2).  index_read=1 / 2: the records of the I1 / I2 file
    instead -- the header of mate `read_no`, the i7 / i5 that header carries as the sequence, and 'F' qualities."""
    if index_read not in (None, 1, 2) or (index_read == 2 and not spec.l2):
        raise ValueError(f"index read {index_read!r} of a spec with l2 = {spec.l2}")
    n = g1 - g0
    if n <= 0:
        return b""
    g = np.arange(g0, g1, dtype=np.uint64)
    cols, valid = [], []

    def const(bs):
        for ch in bs:
            cols.append(np.full(n, ch, np.uint8))
            valid.append(np.ones(n, bool))

    def number(val, max_digits, min_digits):
        val = val.astype(np.int64)
        for d in range(max_digits - 1, -1, -1):
            cols.append((val // 10 ** d % 10 + 48).astype(np.uint8))
            valid.append(np.ones(n, bool) if d < min_digits else (val >= 10 ** d))

    wc = draw(spec.seed, g, J_COORD)
    x = np.uint64(1000) + (wc & np.uint64(0xFFFFFFFF)) % np.uint64(31000)
    y = np.uint64(1000) + (wc >> np.uint64(32)) % np.uint64(199000)
    tile = np.uint64(1101) + g % np.uint64(78)
    const(PREFIX + str(spec.lane).encode() + b":")
    number(tile, 4, 4)
    const(b":")
    number(x, 5, 4)
    const(b":")
    number(y, 6, 4)
    const(b" " + str(read_no).encode() + b":N:0:")
    i7, i5 = index_codes(spec, g)
    for p in range(spec.l1):
        cols.append(SYMS[i7[:, p]]); valid.append(np.ones(n, bool))
    if spec.l2:
        const(b"+")
        for p in range(spec.l2):
            cols.append(SYMS[i5[:, p]]); valid.append(np.ones(n, bool))
    const(b"\n")
    if index_read:
        seq = i7 if index_read == 1 else i5
        for p in range(seq.shape[1]):
            cols.append(SYMS[seq[:, p]]); valid.append(np.ones(n, bool))
        const(b"\n+\n" + b"F" * seq.shape[1] + b"\n")
        return np.stack(cols, axis=1)[np.stack(valid, axis=1)].tobytes()
    j0 = J_SEQ1 if read_no == 1 else J_SEQ2
    words = [draw(spec.seed, g, j0 + k) for k in range((spec.read_len + 31) // 32)]
    for i in range(spec.read_len):
        code = ((words[i // 32] >> np.uint64(2 * (i % 32))) & np.uint64(3)).astype(np.uint8)
        cols.append(BASES[code]); valid.append(np.ones(n, bool))
    const(b"\n+\n" + b"F" * spec.read_len + b"\n")
    mat = np.stack(cols, axis=1)
    msk = np.stack(valid, axis=1)
    return mat[msk].tobytes()


def generate_big(spec, g0, g1, read_no=1, step=200_000, index_read=None):
    """generate() in slices, to bound the temporary matrices."""
    return b"".join(generate(spec, a, min(a + step, g1), read_no, index_read) for a in range(g0, g1, step))


def binned_qualities(data, seed=0):
    """The same FASTQ with every quality symbol drawn from four binned values, as binned Illumina qualities look:
    'F' 85 %, ':' 10 %, ',' 4 %, '#' 1 % (generate() writes all-'F' qualities).  Headers, bases and lengths stay."""
    a = np.frombuffer(data, np.uint8).copy()
    if not a.size:
        return b""
    line = np.empty(a.size, np.uint32)
    line[0] = 0
    np.cumsum(a[:-1] == 10, dtype=np.uint32, out=line[1:])
    qual = (line % 4 == 3) & (a != 10)
    rng = np.random.default_rng(seed)
    a[qual] = rng.choice(np.frombuffer(b"F:,#", np.uint8), int(qual.sum()), p=[0.85, 0.10, 0.04, 0.01])
    return a.tobytes()
