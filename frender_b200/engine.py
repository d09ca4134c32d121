"""Host-side mirror of the reference's hot-path functions over the CUDA library.

Names, argument meaning and error behaviour follow the reference (frender.py, "F:"):
    tally_barcodes(cores, files, sample)            F:183-207
    process(cores, barcode_counter, indexes, n, rc) F:391-426
    call_rc_mode_per_id / second pass               F:354-388, F:618-630  (Context.analyze)
The Python here only marshals: strings <-> packed keys, device arrays <-> dicts.  Every
count, match and classification comes from the kernels; nothing falls back to the CPU.
"""
import os

import numpy as np

from . import _lib
from ._lib import C, FrbError, READ_TYPES, check, lib

MAX_SYMS = 21
MAX_WIDE_SYMS = 2 * MAX_SYMS   # a wide context's keys: (lo, hi), see include/frender_b200.h
_ENC = np.full(256, 255, np.uint8)
for _ch, _code in zip(b"ACGTN+", range(1, 7)):
    _ENC[_ch] = _code
_ENC[0] = 0
_ENC_SHEET = np.full(256, 7, np.uint8)          # sheet symbols outside ACGTN never match a read
for _ch, _code in zip(b"ACGTN+", range(1, 7)):
    _ENC_SHEET[_ch] = _code
    _ENC_SHEET[ord(chr(_ch).lower())] = _code   # matching is case-insensitive (F:226)
_ENC_SHEET[0] = 0
_DEC = np.frombuffer(b"\0ACGTN+?", dtype=np.uint8)
_SHIFTS = (np.arange(MAX_SYMS, dtype=np.uint64) * np.uint64(3))
_RC = str.maketrans("ATGCNatgcn", "TACGNtacgn")


def reverse_complement(seq):
    """F:210-211."""
    return seq.translate(_RC)[::-1]


def pack_keys(strings, sheet_mode=False):
    """list of index strings -> uint64 array (3 bits/symbol, see include/frender_b200.h)."""
    if len(strings) == 0:
        return np.zeros(0, np.uint64)
    raw = [s.encode() if isinstance(s, str) else s for s in strings]
    if max(len(r) for r in raw) > MAX_SYMS:
        raise FrbError(_lib.ERR_KEY_TOO_LONG, "index field longer than 21 symbols")
    mat = np.array(raw, dtype=f"S{MAX_SYMS}").view(np.uint8).reshape(len(raw), MAX_SYMS)
    codes = (_ENC_SHEET if sheet_mode else _ENC)[mat]
    if not sheet_mode and (codes == 255).any():
        raise FrbError(_lib.ERR_BAD_ALPHABET, "index field holds a symbol outside ACGTN+")
    return (codes.astype(np.uint64) << _SHIFTS).sum(axis=1, dtype=np.uint64)


def unpack_keys(keys):
    """uint64 array -> list of str (exact inverse of pack_keys for read keys)."""
    keys = np.asarray(keys, dtype=np.uint64)
    if keys.size == 0:
        return []
    codes = ((keys[:, None] >> _SHIFTS) & np.uint64(7)).astype(np.uint8)
    txt = np.ascontiguousarray(_DEC[codes]).view(f"S{MAX_SYMS}").ravel()
    return [t.decode() for t in txt.tolist()]


def pack_keys2(strings, sheet_mode=False):
    """list of index strings of up to 42 symbols -> (lo, hi) uint64 arrays (wide keys, include/frender_b200.h).
    lo equals pack_keys() for strings of up to 21 symbols, whose hi is 0."""
    if len(strings) == 0:
        return np.zeros(0, np.uint64), np.zeros(0, np.uint64)
    raw = [s.encode() if isinstance(s, str) else s for s in strings]
    if max(len(r) for r in raw) > MAX_WIDE_SYMS:
        raise FrbError(_lib.ERR_KEY_TOO_LONG, f"index field longer than {MAX_WIDE_SYMS} symbols")
    mat = np.array(raw, dtype=f"S{MAX_WIDE_SYMS}").view(np.uint8).reshape(len(raw), MAX_WIDE_SYMS)
    codes = (_ENC_SHEET if sheet_mode else _ENC)[mat]
    if not sheet_mode and (codes == 255).any():
        raise FrbError(_lib.ERR_BAD_ALPHABET, "index field holds a symbol outside ACGTN+")
    codes = codes.astype(np.uint64)
    lo = (codes[:, :MAX_SYMS] << _SHIFTS).sum(axis=1, dtype=np.uint64)
    hi = (codes[:, MAX_SYMS:] << _SHIFTS).sum(axis=1, dtype=np.uint64)
    return lo, hi


def unpack_keys2(lo, hi):
    """(lo, hi) uint64 arrays -> list of str (exact inverse of pack_keys2 for read keys)."""
    lo = np.asarray(lo, dtype=np.uint64)
    hi = np.asarray(hi, dtype=np.uint64)
    if lo.size == 0:
        return []
    codes = np.concatenate([(lo[:, None] >> _SHIFTS) & np.uint64(7), (hi[:, None] >> _SHIFTS) & np.uint64(7)], axis=1)
    txt = np.ascontiguousarray(_DEC[codes.astype(np.uint8)]).view(f"S{MAX_WIDE_SYMS}").ravel()
    return [t.decode() for t in txt.tolist()]


def _ptr(arr):
    return arr.ctypes.data_as(C.c_void_p) if arr is not None else None


class PackedSheet:
    """Sample sheet in the matcher's layout (frb_sheet_load)."""

    def __init__(self, indexes, wide=False):
        self.ids = list(indexes["id"])
        self.idx1 = list(indexes["idx1"])
        self.single = indexes.get("idx2") is None
        self.idx2 = [""] * len(self.ids) if self.single else list(indexes["idx2"])
        self.rc_idx2 = [reverse_complement(s) for s in self.idx2]              # F:315
        n = len(self.ids)
        self.l1 = len(self.idx1[0]) if n else 1
        self.l2 = 0 if self.single else (len(self.idx2[0]) if n else 1)
        # rows of unequal length make every comparison in the reference assert (F:227)
        for a, b in zip(self.idx1, self.idx2):
            if len(a) != self.l1 or len(b) != self.l2:
                raise AssertionError(
                    f"Barcode lengths differ inside the sample sheet ({a!r}/{b!r} vs {self.l1}+{self.l2})")
        join = (lambda a, b: a) if self.single else (lambda a, b: a + "+" + b)
        fwd = [join(a, b) for a, b in zip(self.idx1, self.idx2)]
        rc = [join(a, b) for a, b in zip(self.idx1, self.rc_idx2)]
        self.wide = wide
        if wide:    # rows of up to 21+21 symbols (frb_sheet_load2)
            (self.fwd, self.fwd_hi), (self.rc, self.rc_hi) = pack_keys2(fwd, True), pack_keys2(rc, True)
        else:
            self.fwd, self.rc = pack_keys(fwd, sheet_mode=True), pack_keys(rc, sheet_mode=True)
        first_row = {}
        self.group = np.array([first_row.setdefault(name, len(first_row)) for name in self.ids], np.int32)
        self.group_names = list(first_row)                                     # dict order, F:367


class Context:
    """One GPU context (frb_ctx).  Not thread-safe; use one per GPU."""

    def __init__(self, device=0, table_log2=22, wide=False):
        self._h = C.c_void_p()
        rc = lib.frb_create(device, table_log2, C.byref(self._h))
        if rc != _lib.OK:
            msg = lib.frb_last_error(None)
            raise FrbError(rc, msg.decode() if msg else "")
        self.device = device
        self.table_log2 = table_log2
        self.sheet = None
        self.file_names = []
        self.wide = False
        if wide:
            self.set_wide()

    def set_wide(self, on=True):
        """Keys of up to 42 symbols (128-bit keys, frb_set_key_width).  Forgets every file scanned so far."""
        self._ck(lib.frb_set_key_width(self._h, 128 if on else 64))
        self.wide = bool(on)
        self.sheet = None
        self.file_names = []
        self._sharded = False

    def close(self):
        if self._h:
            lib.frb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        return check(self._h, rc)

    # ---- hot path A -------------------------------------------------------------------------
    def reset(self):
        self._ck(lib.frb_reset(self._h))
        self.file_names = []
        self._sharded = False

    def resize_tables(self, table_log2):
        """New unique-key tables of 2^table_log2 slots; forgets every file scanned so far."""
        self._ck(lib.frb_resize_tables(self._h, table_log2))
        self.table_log2 = table_log2
        self.file_names = []
        self._sharded = False

    def scan_gz(self, path, ordinal, sample=None):
        """One fastq.gz through the inflate -> H2D -> kernel pipeline (scan_file, F:154-181).
        Returns (reads, unique keys, decompressed bytes)."""
        reads, uniq, raw = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_scan_gz(self._h, os.fsencode(str(path)), ordinal, sample or 0,
                                 C.byref(reads), C.byref(uniq), C.byref(raw)))
        self.file_names.append(os.path.basename(str(path)))
        return reads.value, uniq.value, raw.value

    def scan_gz_batch(self, paths, ordinals):
        """A run of small fastq.gz files in one go (frb_scan_gz_batch): [(reads, unique keys, decompressed bytes)]
        per file, as scan_gz would give one by one -- or None when the library declined (scan them one by one).
        ordinals: the files' ordinals, or the first of consecutive ones."""
        n = len(paths)
        if isinstance(ordinals, int):
            ordinals = range(ordinals, ordinals + n)
        ords = np.array(list(ordinals), np.uint32)
        names = (C.c_char_p * n)(*[os.fsencode(str(p)) for p in paths])
        reads, uniq, raw = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)
        used = C.c_int()
        self._ck(lib.frb_scan_gz_batch(self._h, names, _ptr(ords), n, _ptr(reads), _ptr(uniq), _ptr(raw), C.byref(used)))
        if not used.value:
            return None
        self.file_names.extend(os.path.basename(str(p)) for p in paths)
        return list(zip(reads.tolist(), uniq.tolist(), raw.tolist()))

    def gz_inflate(self, path, cap):
        """A .gz file inflated on the device (tests, tools).  Returns the bytes, or None when the device path
        declined the stream (frb_scan_gz then inflates it with zlib on a host thread)."""
        out = np.empty(max(cap, 1), np.uint8)
        n, used = C.c_uint64(), C.c_int()
        self._ck(lib.frb_gz_inflate(self._h, os.fsencode(str(path)), _ptr(out), cap, C.byref(n), C.byref(used)))
        return out[:n.value].tobytes() if used.value else None

    def scan_bytes(self, data, ordinal=0, sample=None, rule=_lib.RULE_SCAN, name=None, chunk=None, line_base=0):
        """Decompressed FASTQ bytes from host memory, optionally fed in `chunk`-sized pieces cut
        at line ends.  line_base: lines of the FILE in front of `data` (a rank that scans only some chunks of a
        file passes each chunk's global line number; `first` then holds global read ordinals and the per-rank
        lists merge exactly, SURVEY 8e).  Returns (reads, unique keys)."""
        self._ck(lib.frb_scan_begin(self._h, ordinal, sample or 0))
        view = memoryview(data)
        pos, n = 0, len(view)
        step = chunk or max(n, 1)
        first = True
        while pos < n:
            end = min(pos + step, n)
            if end < n:
                cut = bytes(view[pos:end]).rfind(b"\n")
                if cut < 0:
                    raise FrbError(_lib.ERR_ARG, "chunk holds no line end")
                end = pos + cut + 1
            piece = np.frombuffer(view[pos:end], dtype=np.uint8)
            self._ck(lib.frb_scan_chunk_host(self._h, _ptr(piece), piece.size, line_base if first else _lib.CARRY, rule))
            first = False
            pos = end
        reads, uniq = C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_scan_end(self._h, C.byref(reads), C.byref(uniq)))
        self.file_names.append(name or f"file{ordinal}")
        return reads.value, uniq.value

    def _export(self, fn, n):
        keys, counts, first = (np.empty(n, np.uint64) for _ in range(3))
        self._ck(fn(_ptr(keys), _ptr(counts), _ptr(first), n))
        return keys, counts, first

    def file_arrays(self, i):
        uniq, reads = C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_file_size(self._h, i, C.byref(uniq), C.byref(reads)))
        return self._export(lambda k, c, f, n: lib.frb_file_export(self._h, i, k, c, f, n), uniq.value)

    def file_keys_hi(self, i):
        """Upper key words of file i, in the order of file_arrays (all zero on a narrow context)."""
        uniq, reads = C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_file_size(self._h, i, C.byref(uniq), C.byref(reads)))
        hi = np.empty(uniq.value, np.uint64)
        self._ck(lib.frb_file_export_hi(self._h, i, _ptr(hi), uniq.value))
        return hi

    def total_keys_hi(self):
        """Upper key words of "total", in the order of total_arrays (all zero on a narrow context)."""
        uniq = C.c_uint64()
        self._ck(lib.frb_total_finish(self._h, C.byref(uniq)))
        hi = np.empty(uniq.value, np.uint64)
        self._ck(lib.frb_total_export_hi(self._h, _ptr(hi), uniq.value))
        return hi

    def key_strings(self, keys, keys_hi=None):
        """Packed keys of this context -> str."""
        return unpack_keys2(keys, keys_hi) if self.wide else unpack_keys(keys)

    def total_arrays(self):
        """(keys, counts, first_pos) of "total", in first-appearance order (F:199-203)."""
        uniq = C.c_uint64()
        self._ck(lib.frb_total_finish(self._h, C.byref(uniq)))
        return self._export(lambda k, c, f, n: lib.frb_total_export(self._h, k, c, f, n), uniq.value)

    def counter(self):
        """The reference's barcode_counter dict: {"total": {...}, basename: {...}} (F:200-207)."""
        keys, counts, _ = self.total_arrays()
        hi = self.total_keys_hi() if self.wide else None
        out = {"total": dict(zip(self.key_strings(keys, hi), counts.tolist()))}
        for i, name in enumerate(self.file_names):
            k, c, _ = self.file_arrays(i)
            hi = self.file_keys_hi(i) if self.wide else None
            out[name] = dict(zip(self.key_strings(k, hi), c.tolist()))      # same basename overwrites, F:205
        return out

    # ---- hot path B -------------------------------------------------------------------------
    def load_sheet(self, indexes):
        sh = indexes if isinstance(indexes, PackedSheet) and indexes.wide == self.wide else PackedSheet(
            indexes if not isinstance(indexes, PackedSheet) else
            {"id": indexes.ids, "idx1": indexes.idx1, "idx2": None if indexes.single else indexes.idx2}, wide=self.wide)
        if self.wide:
            self._ck(lib.frb_sheet_load2(self._h, _ptr(sh.fwd), _ptr(sh.fwd_hi), _ptr(sh.rc), _ptr(sh.rc_hi),
                                         _ptr(sh.group), len(sh.ids), sh.l1, sh.l2))
        else:
            self._ck(lib.frb_sheet_load(self._h, _ptr(sh.fwd), _ptr(sh.rc), _ptr(sh.group), len(sh.ids), sh.l1, sh.l2))
        self.sheet = sh
        return sh

    def load_total(self, counter, single=False):
        """Use a caller-supplied {key: reads} dict as the unique-key list (process(), F:391).
        Only the first two '+' parts of a key take part in matching (F:306)."""
        if single:
            heads = list(counter.keys())
        else:
            heads = []
            for k in counter:
                idx1, idx2 = k.split("+")[0:2]            # ValueError without a '+', as in F:306
                heads.append(idx1 + "+" + idx2)
        counts = np.fromiter(counter.values(), dtype=np.uint64, count=len(counter))
        if self.wide:
            keys, hi = pack_keys2(heads)
            self._ck(lib.frb_total_load2(self._h, _ptr(keys), _ptr(hi), _ptr(counts), len(keys)))
        else:
            keys = pack_keys(heads)
            self._ck(lib.frb_total_load(self._h, _ptr(keys), _ptr(counts), len(keys)))

    def load_total_arrays(self, keys, counts):
        """Use packed key / count arrays as the unique-key list (already in first-appearance order)."""
        keys = np.ascontiguousarray(keys, np.uint64)
        counts = np.ascontiguousarray(counts, np.uint64)
        self._ck(lib.frb_total_load(self._h, _ptr(keys), _ptr(counts), len(keys)))

    def merge_list(self, keys, counts, first_pos):
        """Fold a (key, count, global first_pos) list from another context into this context's total."""
        keys, counts, first_pos = (np.ascontiguousarray(x, np.uint64) for x in (keys, counts, first_pos))
        self._ck(lib.frb_total_merge(self._h, _ptr(keys), _ptr(counts), _ptr(first_pos), len(keys)))

    # ---- multi-GPU ----------------------------------------------------------------------------
    @staticmethod
    def nccl_unique_id():
        ident = (C.c_char * 128)()
        rc = lib.frb_nccl_unique_id(ident)
        if rc != _lib.OK:
            raise FrbError(rc, (lib.frb_last_error(None) or b"").decode())
        return bytes(ident)

    def nccl_init(self, ident, rank, n_ranks):
        self._ck(lib.frb_nccl_init(self._h, ident, rank, n_ranks))

    def allmerge(self):
        """Merge the per-rank totals over NCCL; every rank ends with the same total list."""
        n = C.c_uint64()
        self._ck(lib.frb_allmerge(self._h, C.byref(n)))
        self._sharded = False
        return n.value

    def shardmerge(self):
        """Merge the per-rank totals over NCCL so that every key ends on one rank (its owner by hash):
        this rank's total becomes its share of the job-wide total.  Returns the size of the share."""
        n = C.c_uint64()
        self._ck(lib.frb_shardmerge(self._h, C.byref(n)))
        self._sharded = True
        return n.value

    def allreduce(self, arr):
        """Element-wise sum of a small uint64 array over all ranks."""
        arr = np.ascontiguousarray(arr, np.uint64).copy()
        self._ck(lib.frb_allreduce_u64(self._h, _ptr(arr), arr.size))
        return arr

    def match(self, n_subs, rc_mode, use_rc_rows=None, want_outputs=True):
        """Raw matcher call over the context's total list.  Returns a dict of numpy arrays."""
        uniq = C.c_uint64()
        self._ck(lib.frb_total_finish(self._h, C.byref(uniq)))
        n, rows = uniq.value, len(self.sheet.ids)
        out = {}
        if want_outputs:
            out = {"m1": np.empty(n, np.int32), "m2": np.empty(n, np.int32), "type": np.empty(n, np.uint8),
                   "srow": np.empty(n, np.int32)}
            if rc_mode:
                out.update({"m2rc": np.empty(n, np.int32), "type_rc": np.empty(n, np.uint8),
                            "srow_rc": np.empty(n, np.int32)})
        out["f_sum"] = np.zeros(max(rows, 1), np.uint64)
        out["rc_sum"] = np.zeros(max(rows, 1), np.uint64)
        use = None if use_rc_rows is None else np.ascontiguousarray(use_rc_rows, dtype=np.uint8)
        try:
            self._ck(lib.frb_match(self._h, n_subs, 1 if rc_mode else 0, _ptr(use), _ptr(out.get("m1")),
                                   _ptr(out.get("m2")), _ptr(out.get("type")), _ptr(out.get("srow")),
                                   _ptr(out.get("m2rc")), _ptr(out.get("type_rc")), _ptr(out.get("srow_rc")),
                                   _ptr(out["f_sum"]), _ptr(out["rc_sum"])))
        except FrbError as exc:
            if exc.code == _lib.ERR_BAD_LENGTH:      # the reference asserts / fails to unpack here
                raise AssertionError(exc.message) from None
            raise
        return out

    def process(self, counter, indexes, num_subs, rc_mode, use_rc_rows=None):
        """{key: {...}} exactly as the reference's process() returns it (F:391-426)."""
        sh = self.load_sheet(indexes)
        if counter is not None:
            self.load_total(counter, single=sh.single)
        keys, counts, _ = self.total_arrays()
        names = list(counter.keys()) if counter is not None else self.key_strings(
            keys, self.total_keys_hi() if self.wide else None)
        r = self.match(num_subs, rc_mode, use_rc_rows)
        idx2 = sh.idx2
        if use_rc_rows is not None:
            idx2 = [b if u else a for a, b, u in zip(sh.idx2, sh.rc_idx2, use_rc_rows)]
        pick = lambda table, rows: [table[i] if i >= 0 else "" for i in rows.tolist()]
        cols = {"matched_idx1": pick(sh.idx1, r["m1"]), "matched_idx2": pick(idx2, r["m2"]),
                "read_type": [READ_TYPES[t] for t in r["type"].tolist()],
                "sample_name": pick(sh.ids, r["srow"]), "reads": counts.tolist()}
        if rc_mode:
            cols["matched_rc_idx2"] = pick(sh.rc_idx2, r["m2rc"])
            cols["rc_read_type"] = [READ_TYPES[t] for t in r["type_rc"].tolist()]
            cols["rc_sample_name"] = pick(sh.ids, r["srow_rc"])
        fields = list(cols)
        return {name: dict(zip(fields, vals)) for name, vals in zip(names, zip(*cols.values()))}, r

    def rc_calls(self, match_out):
        """call_rc_mode_per_id (F:354-388) from the device's per-name sums."""
        sh = self.sheet
        calls = {}
        for g, name in enumerate(sh.group_names):
            f, r = int(match_out["f_sum"][g]), int(match_out["rc_sum"][g])
            calls[name] = {"call": f < r, "reads_f": f, "reads_rc": r}
        return calls

    def analyze(self, indexes, num_subs, rc_mode, counter=None):
        """Matcher part of frender_scan (F:610-630).  Returns (results, rc_calls, oriented idx2)."""
        results, raw = self.process(counter, indexes, num_subs, rc_mode)
        if not rc_mode:
            return results, None, list(self.sheet.idx2)
        if getattr(self, "_sharded", False):   # the orientation call is over all reads of the job (F:354-388)
            raw = dict(raw, f_sum=self.allreduce(raw["f_sum"]), rc_sum=self.allreduce(raw["rc_sum"]))
        calls = self.rc_calls(raw)
        use = np.array([calls[name]["call"] for name in self.sheet.ids], np.uint8)      # F:618-623
        oriented = [b if u else a for a, b, u in zip(self.sheet.idx2, self.sheet.rc_idx2, use)]
        results, _ = self.process(None, indexes, num_subs, False, use_rc_rows=use)
        return results, calls, oriented

    # ---- hot path C -------------------------------------------------------------------------
    def demux_ok(self, match, file_lists=None):
        """demux_ok per unique key of the total list (in export order) and a flag per file that holds a key it
        should not (frb_demux_ok; F:504-564).  match: uint8 [(4 + sheet rows), n_files] class x file matrix (0 no,
        1 yes, 2 invalid pattern).  file_lists: None = the per-file lists of this context, else [(keys, counts)]
        host arrays.  Returns (ok bool array, bad-file bool array, offending sample row or None)."""
        match = np.ascontiguousarray(match, np.uint8)
        n_files = match.shape[1]
        n = C.c_uint64()
        self._ck(lib.frb_total_finish(self._h, C.byref(n)))
        ok, bad = np.ones(max(n.value, 1), np.uint8), np.zeros(max(n_files, 1), np.uint8)
        err = C.c_int32()
        if file_lists is None:
            kp = cp = np_ = None
        else:
            keep = [(np.ascontiguousarray(k, np.uint64), np.ascontiguousarray(c, np.uint64)) for k, c in file_lists]
            kp = (C.c_void_p * n_files)(*[k.ctypes.data for k, _ in keep])
            cp = (C.c_void_p * n_files)(*[c.ctypes.data for _, c in keep])
            np_ = (C.c_uint64 * n_files)(*[k.size for k, _ in keep])
        self._ck(lib.frb_demux_ok(self._h, _ptr(match), n_files, kp, cp, np_, _ptr(ok), _ptr(bad), C.byref(err)))
        return ok[:n.value].astype(bool), bad[:n_files].astype(bool), (None if err.value == 0x7FFFFFFF else err.value)

    def route_load(self, keys, sink_ids, n_sinks, keys_hi=None):
        """Results table for the demux router: packed key -> sink id (unique keys).  keys_hi: upper words of a wide
        context's keys (pack_keys2)."""
        keys = np.ascontiguousarray(keys, np.uint64)
        sink_ids = np.ascontiguousarray(sink_ids, np.uint32)
        if keys_hi is None:
            self._ck(lib.frb_route_load(self._h, _ptr(keys), _ptr(sink_ids), len(keys), n_sinks))
        else:
            hi = np.ascontiguousarray(keys_hi, np.uint64)
            self._ck(lib.frb_route_load2(self._h, _ptr(keys), _ptr(hi), _ptr(sink_ids), len(keys), n_sinks))
        self._n_sinks = n_sinks

    def route_pair(self, r1, r2, final=3):
        """Partition one record-aligned chunk pair by sink (frb_route_pair).  Returns
        (out_r1, out_r2, off_r1, off_r2, pairs, consumed_r1, consumed_r2); sink s of mate m is
        out_m[off_m[s]:off_m[s+1]]."""
        a = np.frombuffer(r1, np.uint8)
        b = np.frombuffer(r2, np.uint8)
        o1, o2 = np.empty(max(a.size, 1), np.uint8), np.empty(max(b.size, 1), np.uint8)
        off1, off2 = np.zeros(self._n_sinks + 1, np.uint64), np.zeros(self._n_sinks + 1, np.uint64)
        pairs, u1, u2, bad = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_route_pair(self._h, _ptr(a), a.size, _ptr(b), b.size, int(final), _ptr(o1), _ptr(o2),
                                    _ptr(off1), _ptr(off2), C.byref(pairs), C.byref(u1), C.byref(u2), C.byref(bad)))
        return (o1[:u1.value].tobytes(), o2[:u2.value].tobytes(), off1.astype(np.int64), off2.astype(np.int64),
                pairs.value, u1.value, u2.value)

    def route_reset(self, chunk_bytes=None):
        """A new stream of chunk pairs begins (frb_route_reset); chunk_bytes: the largest chunk per mate that will
        be pushed (frb_route_reserve) -- without it the first chunk sets the size."""
        if chunk_bytes:
            self._ck(lib.frb_route_reserve(self._h, int(chunk_bytes)))
        else:
            self._ck(lib.frb_route_reset(self._h))

    def route_push(self, r1, r2, final=0):
        """Queue one chunk pair of the demux stream (frb_route_push): bytes cut anywhere; what is not complete
        yet is carried on the device.  Returns at once; at most two chunks may be in flight."""
        a = np.frombuffer(r1, np.uint8)
        b = np.frombuffer(r2, np.uint8)
        self._ck(lib.frb_route_push(self._h, _ptr(a), a.size, _ptr(b), b.size, int(final)))

    def route_pop(self):
        """The oldest chunk in flight (frb_route_pop): (out_r1, out_r2, off_r1, off_r2, pairs, carry_r1, carry_r2).
        out_m are views of the library's pinned memory, valid until the chunk after next is pushed; sink s of
        mate m is out_m[off_m[s]:off_m[s+1]]."""
        o1, o2 = C.c_void_p(), C.c_void_p()
        off1, off2 = np.zeros(self._n_sinks + 1, np.uint64), np.zeros(self._n_sinks + 1, np.uint64)
        pairs, c1, c2, bad = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._ck(lib.frb_route_pop(self._h, C.byref(o1), C.byref(o2), _ptr(off1), _ptr(off2), C.byref(pairs),
                                   C.byref(c1), C.byref(c2), C.byref(bad)))
        n1, n2 = int(off1[-1]), int(off2[-1])
        v1 = np.ctypeslib.as_array((C.c_uint8 * max(n1, 1)).from_address(o1.value))[:n1]
        v2 = np.ctypeslib.as_array((C.c_uint8 * max(n2, 1)).from_address(o2.value))[:n2]
        return v1, v2, off1.astype(np.int64), off2.astype(np.int64), pairs.value, c1.value, c2.value

    # ---- measurement ------------------------------------------------------------------------
    def launches(self):
        return lib.frb_launch_count(self._h)

    def prof(self, on=True):
        self._ck(lib.frb_prof_enable(self._h, 1 if on else 0))

    def prof_read(self, kclass, reset=True):
        ms, n = C.c_double(), C.c_uint64()
        self._ck(lib.frb_prof_read(self._h, kclass, C.byref(ms), C.byref(n), 1 if reset else 0))
        return ms.value, n.value


_default = None


def default_context():
    global _default
    if _default is None:
        _default = Context()
    return _default


def tally_barcodes(cores, files, sample=None, ctx=None):
    """Drop-in for the reference's tally_barcodes (F:183-207).  `cores` is accepted for
    signature compatibility; parallelism comes from the GPU, not from a process pool."""
    ctx = ctx or default_context()
    if sample:
        assert sample >= 1, "Number of reads to sample must be ≥ 1!"
    ctx.reset()
    try:
        for ordinal, path in enumerate(files):
            ctx.scan_gz(path, ordinal, sample)
    except FrbError as exc:
        if exc.code != _lib.ERR_KEY_TOO_LONG or ctx.wide:
            raise
        # a dict never refuses a key (F:172-177): index fields longer than 21 symbols take 128-bit keys
        ctx.set_wide()
        for ordinal, path in enumerate(files):
            ctx.scan_gz(path, ordinal, sample)
    return ctx.counter()


def process(cores, barcode_counter, indexes, num_subs, rc_mode, ctx=None):
    """Drop-in for the reference's process (F:391-426)."""
    ctx = ctx or default_context()
    return ctx.process(barcode_counter, indexes, num_subs, rc_mode)[0]
