"""Wide (128-bit) keys on the host: packing, its C-ABI twin and the CSV writer.  No GPU needed."""
import csv
import ctypes as C
import io
import random

import numpy as np
import pytest

import frender_b200._lib as L
from frender_b200.engine import FrbError, pack_keys, pack_keys2, unpack_keys2

SYMS = "ACGTN+"


def rand_key(rng, n):
    return "".join(rng.choice(SYMS) for _ in range(n))


def test_pack_keys2_roundtrip_0_to_42():
    rng = random.Random(7)
    keys = [rand_key(rng, n) for n in range(43) for _ in range(3)]
    lo, hi = pack_keys2(keys)
    assert unpack_keys2(lo, hi) == keys
    assert not (lo >> np.uint64(63)).any()           # bit 63 of lo stays free (FRB_EMPTY_KEY)
    short = [k for k in keys if len(k) <= 21]
    lo_s, hi_s = pack_keys2(short)
    assert (hi_s == 0).all() and (lo_s == pack_keys(short)).all()
    with pytest.raises(FrbError) as e:
        pack_keys2(["A" * 43])
    assert e.value.code == L.ERR_KEY_TOO_LONG


def test_c_abi_pack_key2_matches_python():
    rng = random.Random(11)
    lo, hi = C.c_uint64(), C.c_uint64()
    buf = C.create_string_buffer(44)
    for n in range(43):
        key = rand_key(rng, n)
        assert L.lib.frb_pack_key2(key.encode(), n, 0, C.byref(lo), C.byref(hi)) == L.OK
        plo, phi = pack_keys2([key])
        assert (lo.value, hi.value) == (int(plo[0]), int(phi[0]))
        assert L.lib.frb_unpack_key2(lo, hi, buf) == n
        assert buf.value.decode() == key
    assert L.lib.frb_pack_key2(b"A" * 43, 43, 0, C.byref(lo), C.byref(hi)) == L.ERR_KEY_TOO_LONG
    assert L.lib.frb_pack_key2(b"ACGX", 4, 0, C.byref(lo), C.byref(hi)) == L.ERR_BAD_ALPHABET


def test_write_scan_csv2_bytes(tmp_path):
    rng = random.Random(3)
    keys = []
    for n in (1, 10, 21, 25, 30, 42):
        a = rand_key(random.Random(n), n // 2).replace("+", "A")
        keys.append(a + "+" + rand_key(rng, n - len(a) - 1).replace("+", "C") if n > len(a) else a)
    keys += ["ACGTACGTACGT+TTGGCCAATTGG", "A" * 20 + "+" + "C" * 21, "ACGT" * 10 + "AA"]
    lo, hi = pack_keys2(keys)
    n = len(keys)
    counts = np.arange(1, n + 1, dtype=np.uint64) * 7
    m1 = np.array([0 if i % 2 else -1 for i in range(n)], np.int32)
    m2 = np.array([1 if i % 3 else -1 for i in range(n)], np.int32)
    typ = np.array([i % 4 for i in range(n)], np.uint8)
    srow = np.array([1 if i % 4 == 2 else -1 for i in range(n)], np.int32)
    ok = np.array([i % 2 for i in range(n)], np.uint8)
    idx1, idx2, ids = ["ACGTACGTACGT", "TTTTTTTTTTTT"], ["GGGGGGGGGGGG", "CC,AA"], ["S1", 'S"2']
    strs = lambda items: (C.c_char_p * len(items))(*[s.encode() for s in items])
    path = tmp_path / "out.csv"
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = L.lib.frb_write_scan_csv2(str(path).encode(), p(lo), p(hi), p(counts), p(m1), p(m2), p(typ), p(srow), p(ok),
                                   n, strs(idx1), strs(idx2), strs(ids), 2, 0)
    assert rc == L.OK
    buf = io.StringIO(newline="")
    w = csv.writer(buf)
    w.writerow(["idx1", "idx2", "matched_idx1", "matched_idx2", "read_type", "sample_name", "reads", "demux_ok"])
    for i, k in enumerate(keys):
        parts = k.split("+")
        w.writerow([parts[0], parts[1] if len(parts) > 1 else "", idx1[m1[i]] if m1[i] >= 0 else "",
                    idx2[m2[i]] if m2[i] >= 0 else "", L.READ_TYPES[typ[i]], ids[srow[i]] if srow[i] >= 0 else "",
                    int(counts[i]), "True" if ok[i] else "False"])
    assert path.read_bytes() == buf.getvalue().encode()
