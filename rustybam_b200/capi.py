"""ctypes binding of include/rbcuda.h (librbcuda.so).

Used by the tests, bench.py and __graft_entry__; the production host is the C++ `rb` binary /
the Rust shim shown in INTEGRATION.md.  There is no Python or CPU implementation of the path
behind this module: if the CUDA library is missing or no sm_100 device is present, calls raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RBCUDA_LIB") or os.path.join(HERE, "librbcuda.so")  # (RBCUDA_LIB: tuning builds, tools/variants.sh)

RB_OK = 0
RB_ERR_NO_DEVICE, RB_ERR_CUDA, RB_ERR_BAD_ARG = -1, -2, -3
RB_ERR_REF_CIGAR_PARSE, RB_ERR_REF_INTEGRITY, RB_ERR_REF_STRIP, RB_ERR_REF_INDEX = -4, -5, -6, -7
RB_ERR_UNSUPPORTED, RB_ERR_OOM = -8, -9
RB_ERR_REF_PAF_PARSE = -10
REF_PANIC_CODES = (RB_ERR_REF_CIGAR_PARSE, RB_ERR_REF_INTEGRITY, RB_ERR_REF_STRIP, RB_ERR_REF_INDEX)
POLICY_RIGHTMOST, POLICY_EARLY_EXIT = 0, 1
WANT_TEXT, WANT_NUMERIC, WANT_QBED, WANT_STATS_TEXT = 1, 2, 4, 8
LIFT_SEARCH, LIFT_STREAM = 0, 1

EXPORTS = [
    "rb_ctx_create", "rb_ctx_destroy", "rb_last_error", "rb_ctx_set_stream", "rb_ctx_set_profiling", "rb_ctx_set_lift_mode", "rb_ctx_set_slicing", "rb_ctx_kernel_times",
    "rb_liftover", "rb_stats", "rb_break_paf", "rb_invert", "rb_trim_paf", "rb_trim_paf_begin", "rb_trim_paf_round", "rb_trim_paf_end", "rb_batch_break", "rb_free_lift_out", "rb_free_stats_out", "rb_batch_upload", "rb_batch_liftover", "rb_batch_stats",
    "rb_batch_download_lift", "rb_batch_download_stats", "rb_batch_free", "rb_sort_windows", "rb_version", "rb_host_register",
    "rb_host_unregister", "rb_is_bgzf", "rb_inflate_bgzf", "rb_free_text", "rb_batch_upload_paf", "rb_batch_set_windows", "rb_batch_records",
    "rb_batch_set_windows_bed", "rb_batch_windows", "rb_liftover_text", "rb_stats_text",
]

u8p, u32p, u64p, f32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_float)


class RbRecords(C.Structure):
    _fields_ = [("n_rec", C.c_uint32), ("cigar", u8p), ("cigar_nbytes", C.c_uint64), ("cigar_off", u64p), ("q_len", u64p),
                ("q_st", u64p), ("q_en", u64p), ("t_len", u64p), ("t_st", u64p), ("t_en", u64p), ("mapq", u64p), ("strand", u8p),
                ("q_id", u32p), ("t_id", u32p), ("names", u8p), ("names_off", u64p), ("n_names", C.c_uint32)]


class RbWindows(C.Structure):
    _fields_ = [("n_win", C.c_uint32), ("t_id", u32p), ("st", u64p), ("en", u64p), ("bed_row", u32p), ("ids", u8p), ("ids_off", u64p)]


class RbLiftOut(C.Structure):
    _fields_ = [("n_out", C.c_uint64), ("paf_text", u8p), ("paf_nbytes", C.c_uint64), ("line_off", u64p), ("q_st", u64p),
                ("q_en", u64p), ("t_st", u64p), ("t_en", u64p), ("nmatch", u64p), ("aln_len", u64p), ("rec_idx", u32p),
                ("win_idx", u32p), ("n_pairs", C.c_uint64), ("_owner", C.c_void_p)]


class RbStatsOut(C.Structure):
    _fields_ = [("n", C.c_uint64), ("equal", u32p), ("diff", u32p), ("ins", u32p), ("del_", u32p), ("ins_events", u32p),
                ("del_events", u32p), ("matches", u32p), ("id_by_matches", f32p), ("id_by_events", f32p), ("id_by_all", f32p),
                ("_owner", C.c_void_p)]


class RbSummary(C.Structure):
    _fields_ = [("n_ops", C.c_uint64), ("n_pairs", C.c_uint64), ("n_out", C.c_uint64), ("out_bytes", C.c_uint64),
                ("cigar_bytes", C.c_uint64)]


class RbPafInfo(C.Structure):
    _fields_ = [("text_bytes", C.c_uint64), ("n_lines", C.c_uint64), ("skipped", C.c_uint64), ("n_rec", C.c_uint32), ("n_names", C.c_uint32),
                ("names", u8p), ("names_off", u64p), ("cigar_bytes", C.c_uint64)]


class RbBedInfo(C.Structure):
    _fields_ = [("text_bytes", C.c_uint64), ("n_lines", C.c_uint64), ("n_comments", C.c_uint64), ("n_parsed", C.c_uint64),
                ("n_win", C.c_uint32), ("n_fields", C.c_uint32), ("default_ids", C.c_int), ("general", C.c_int)]


class RbKernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_uint64), ("ms", C.c_double)]


class RbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rbcuda error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Loads librbcuda.so; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -m rustybam_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.rb_ctx_create.restype = C.c_void_p
    lib.rb_ctx_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]
    lib.rb_ctx_destroy.argtypes = [C.c_void_p]
    lib.rb_last_error.restype = C.c_char_p
    lib.rb_last_error.argtypes = [C.c_void_p]
    lib.rb_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.rb_ctx_set_profiling.argtypes = [C.c_void_p, C.c_int]
    lib.rb_ctx_set_lift_mode.argtypes = [C.c_void_p, C.c_int]
    lib.rb_ctx_set_slicing.argtypes = [C.c_void_p, C.c_uint64]
    lib.rb_ctx_kernel_times.argtypes = [C.c_void_p, C.POINTER(RbKernelTime), C.c_int, C.c_int]
    lib.rb_liftover.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.POINTER(RbWindows), C.c_int, C.c_uint32, C.POINTER(RbLiftOut),
                                C.POINTER(RbStatsOut)]
    lib.rb_stats.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.POINTER(RbStatsOut)]
    lib.rb_break_paf.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.c_uint32, C.c_int, C.c_uint32, C.POINTER(RbLiftOut), C.POINTER(RbStatsOut)]
    lib.rb_invert.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.c_uint32, C.POINTER(RbLiftOut)]
    lib.rb_trim_paf.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(RbLiftOut),
                                C.POINTER(RbStatsOut)]
    lib.rb_trim_paf_begin.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.rb_trim_paf_round.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    lib.rb_trim_paf_end.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.POINTER(RbLiftOut), C.POINTER(RbStatsOut)]
    lib.rb_batch_break.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.c_int, C.POINTER(RbSummary)]
    lib.rb_free_lift_out.argtypes = [C.c_void_p, C.POINTER(RbLiftOut)]
    lib.rb_free_stats_out.argtypes = [C.c_void_p, C.POINTER(RbStatsOut)]
    lib.rb_batch_upload.restype = C.c_void_p
    lib.rb_batch_upload.argtypes = [C.c_void_p, C.POINTER(RbRecords), C.POINTER(RbWindows), C.POINTER(C.c_int)]
    lib.rb_batch_liftover.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_int, C.POINTER(RbSummary)]
    lib.rb_batch_stats.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(RbSummary)]
    lib.rb_batch_download_lift.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(RbLiftOut), C.POINTER(RbStatsOut)]
    lib.rb_batch_download_stats.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(RbStatsOut)]
    lib.rb_batch_free.argtypes = [C.c_void_p, C.c_void_p]
    lib.rb_sort_windows.argtypes = [C.c_uint32, u32p, u64p, u32p]
    lib.rb_version.restype = C.c_char_p
    lib.rb_is_bgzf.argtypes = [C.c_char_p, C.c_uint64]
    lib.rb_inflate_bgzf.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    lib.rb_free_text.argtypes = [C.c_void_p, C.c_void_p]
    lib.rb_batch_upload_paf.restype = C.c_void_p
    lib.rb_batch_upload_paf.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.POINTER(RbPafInfo), C.POINTER(C.c_int)]
    lib.rb_batch_set_windows.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(RbWindows)]
    lib.rb_batch_records.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(RbRecords)]
    lib.rb_batch_set_windows_bed.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint64, C.POINTER(RbBedInfo)]
    lib.rb_batch_windows.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(RbWindows)]
    lib.rb_liftover_text.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p, C.c_uint64, C.c_int, C.c_uint32, C.POINTER(RbLiftOut),
                                     C.POINTER(RbStatsOut), C.POINTER(RbPafInfo), C.POINTER(RbBedInfo)]
    lib.rb_stats_text.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64, C.c_int, C.c_uint32, C.POINTER(RbLiftOut), C.POINTER(RbStatsOut),
                                  C.POINTER(RbPafInfo)]
    lib.rb_host_register.argtypes = [C.c_void_p, C.c_uint64]
    lib.rb_host_unregister.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def _ptr(a, t):
    return a.ctypes.data_as(t)


class Records:
    """Packed SoA records (rb_records).  Keeps the numpy arrays alive next to the C struct."""

    def __init__(self, cigar, cigar_off, q_len, q_st, q_en, t_len, t_st, t_en, mapq, strand, q_id, t_id, names):
        self.cigar = np.ascontiguousarray(cigar, dtype=np.uint8)
        self.cigar_off = np.ascontiguousarray(cigar_off, dtype=np.uint64)
        self.cols = [np.ascontiguousarray(x, dtype=np.uint64) for x in (q_len, q_st, q_en, t_len, t_st, t_en, mapq)]
        self.strand = np.ascontiguousarray(strand, dtype=np.uint8)
        self.q_id = np.ascontiguousarray(q_id, dtype=np.uint32)
        self.t_id = np.ascontiguousarray(t_id, dtype=np.uint32)
        self.names = [n if isinstance(n, bytes) else n.encode() for n in names]
        blob = b"".join(self.names)
        self.names_blob = np.frombuffer(blob + b"\0", dtype=np.uint8).copy()
        self.names_off = np.zeros(len(self.names) + 1, dtype=np.uint64)
        if self.names:
            self.names_off[1:] = np.cumsum([len(n) for n in self.names], dtype=np.uint64)
        n = len(self.q_id)
        self.n_rec = n
        s = RbRecords()
        s.n_rec = n
        s.cigar = _ptr(self.cigar, u8p) if len(self.cigar) else None
        s.cigar_nbytes = int(self.cigar_off[-1]) if len(self.cigar_off) else 0
        s.cigar_off = _ptr(self.cigar_off, u64p)
        (s.q_len, s.q_st, s.q_en, s.t_len, s.t_st, s.t_en, s.mapq) = [_ptr(c, u64p) for c in self.cols]
        s.strand = _ptr(self.strand, u8p)
        s.q_id, s.t_id = _ptr(self.q_id, u32p), _ptr(self.t_id, u32p)
        s.names, s.names_off, s.n_names = _ptr(self.names_blob, u8p), _ptr(self.names_off, u64p), len(self.names)
        self.c = s

    @property
    def cigar_nbytes(self):
        return int(self.c.cigar_nbytes)


class Windows:
    """rb_windows: sorts BED rows by (t_id, st) with rb_sort_windows and keeps bed_row."""

    def __init__(self, t_id, st, en, ids):
        lib = load()
        t_id = np.ascontiguousarray(t_id, dtype=np.uint32)
        st = np.ascontiguousarray(st, dtype=np.uint64)
        en = np.ascontiguousarray(en, dtype=np.uint64)
        n = len(t_id)
        perm = np.zeros(n, dtype=np.uint32)
        rc = lib.rb_sort_windows(n, _ptr(t_id, u32p), _ptr(st, u64p), _ptr(perm, u32p))
        assert rc == 0
        self.t_id, self.st, self.en, self.bed_row = t_id[perm].copy(), st[perm].copy(), en[perm].copy(), perm
        s = RbWindows()
        s.n_win = n
        s.t_id, s.st, s.en = _ptr(self.t_id, u32p), _ptr(self.st, u64p), _ptr(self.en, u64p)
        s.bed_row = _ptr(self.bed_row, u32p)
        if ids is None:  # default ids: formatted on the device
            s.ids, s.ids_off = None, None
        else:
            ids = [i if isinstance(i, bytes) else i.encode() for i in ids]
            ids = [ids[j] for j in perm]
            self.ids_blob = np.frombuffer(b"".join(ids) + b"\0", dtype=np.uint8).copy()
            self.ids_off = np.zeros(n + 1, dtype=np.uint64)
            if n:
                self.ids_off[1:] = np.cumsum([len(i) for i in ids], dtype=np.uint64)
            s.ids, s.ids_off = _ptr(self.ids_blob, u8p), _ptr(self.ids_off, u64p)
        self.c = s
        self.n_win = n


def _np(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


def _paf_info(pi):
    nn = int(pi.n_names)
    off = _np(pi.names_off, nn + 1, np.uint64) if pi.names_off else np.zeros(1, np.uint64)
    blob = C.string_at(pi.names, int(off[-1])) if nn and int(off[-1]) else b""
    return dict(names=[blob[int(off[i]):int(off[i + 1])] for i in range(nn)], n_rec=int(pi.n_rec), n_lines=int(pi.n_lines),
                skipped=int(pi.skipped), text_bytes=int(pi.text_bytes), cigar_bytes=int(pi.cigar_bytes))


class Context:
    """rb_ctx.  One per GPU; not thread-safe (one calling thread per context)."""

    def __init__(self, device=0, devices=None):
        """devices=[d0, d1, ...]: a multi-device context — rb_liftover / rb_stats spread the records over the GPUs and merge
        the rows into one output (the same id may be listed twice: two contexts on one GPU)."""
        self.lib = load()
        st = C.c_int(0)
        ids = list(devices) if devices else [device]
        dev = (C.c_int * len(ids))(*ids)
        self.h = self.lib.rb_ctx_create(dev, len(ids), C.byref(st))
        if not self.h:
            raise RbError(st.value, "rb_ctx_create failed (no sm_100 device? there is no CPU fallback)")

    def close(self):
        if self.h:
            self.lib.rb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != RB_OK:
            raise RbError(rc, self.lib.rb_last_error(self.h).decode())

    def set_stream(self, cuda_stream_ptr):
        self._check(self.lib.rb_ctx_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def set_lift_mode(self, mode):
        self._check(self.lib.rb_ctx_set_lift_mode(self.h, int(mode)))

    def set_slicing(self, min_slice_bytes=16 << 20):
        self._check(self.lib.rb_ctx_set_slicing(self.h, int(min_slice_bytes)))

    def set_profiling(self, on=True):
        self._check(self.lib.rb_ctx_set_profiling(self.h, int(on)))

    def kernel_times(self, reset=True):
        arr = (RbKernelTime * 32)()
        n = self.lib.rb_ctx_kernel_times(self.h, arr, 32, int(reset))
        return {arr[i].name.decode(): (int(arr[i].launches), float(arr[i].ms)) for i in range(min(n, 32))}

    # ---- drop-in calls (host buffers in, pinned host buffers out) ----
    def liftover(self, recs: Records, wins: Windows, policy=POLICY_RIGHTMOST, want=WANT_TEXT | WANT_NUMERIC, stats=True, copy=True):
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_liftover(self.h, C.byref(recs.c), C.byref(wins.c), policy, want, C.byref(out),
                                         C.byref(st) if stats else None))
        res = self._collect_lift(out, st if stats else None, (want & ~WANT_QBED) | (WANT_TEXT if want & WANT_STATS_TEXT else 0)) if copy else dict(n_out=int(out.n_out), paf_nbytes=int(out.paf_nbytes), n_pairs=int(out.n_pairs))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def liftover_view(self, recs: Records, wins: Windows, policy=POLICY_RIGHTMOST, want=WANT_TEXT | WANT_NUMERIC, stats=True):
        """rb_liftover without copying the outputs: returns (views, release) — numpy views straight onto the library's pinned
        block ("paf_text" as a uint8 array), valid until release() is called.  For outputs of many GB (bench.py's checks)."""
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_liftover(self.h, C.byref(recs.c), C.byref(wins.c), policy, want, C.byref(out),
                                         C.byref(st) if stats else None))
        return self._lift_views(out, st, want, stats)

    def _lift_views(self, out, st, want, stats):
        n, nb = int(out.n_out), int(out.paf_nbytes)

        def view(ptr, cnt, dt):
            if not ptr or cnt == 0:
                return np.zeros(0, dtype=dt)
            return np.ctypeslib.as_array(ptr, shape=(cnt,))
        res = dict(n_out=n, n_pairs=int(out.n_pairs), paf_nbytes=nb)
        if want & (WANT_TEXT | WANT_STATS_TEXT):
            res["paf_text"], res["line_off"] = view(out.paf_text, nb, np.uint8), view(out.line_off, n + 1, np.uint64)
        if want & WANT_NUMERIC:
            for k in ("q_st", "q_en", "t_st", "t_en", "nmatch", "aln_len"):
                res[k] = view(getattr(out, k), n, np.uint64)
            res["rec_idx"], res["win_idx"] = view(out.rec_idx, n, np.uint32), view(out.win_idx, n, np.uint32)
        if stats:
            res["stats"] = dict(n=n, equal=view(st.equal, n, np.uint32), diff=view(st.diff, n, np.uint32), ins=view(st.ins, n, np.uint32),
                                **{"del": view(st.del_, n, np.uint32)}, ins_events=view(st.ins_events, n, np.uint32),
                                del_events=view(st.del_events, n, np.uint32), matches=view(st.matches, n, np.uint32),
                                id_by_matches=view(st.id_by_matches, n, np.float32), id_by_events=view(st.id_by_events, n, np.float32),
                                id_by_all=view(st.id_by_all, n, np.float32))

        def release():
            self.lib.rb_free_lift_out(self.h, C.byref(out))
            if stats:
                self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res, release

    def break_paf(self, recs: Records, max_size=100, policy=POLICY_RIGHTMOST, want=WANT_TEXT | WANT_NUMERIC, stats=True, copy=True):
        """rb_break_paf: every record cut at its indels longer than max_size (liftover.rs:182-226), rows in file order."""
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_break_paf(self.h, C.byref(recs.c), max_size, policy, want, C.byref(out), C.byref(st) if stats else None))
        res = self._collect_lift(out, st if stats else None, want) if copy else dict(n_out=int(out.n_out), paf_nbytes=int(out.paf_nbytes), n_pairs=int(out.n_pairs))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def trim_paf(self, recs: Records, match_score=1, diff_score=1, indel_score=1, remove_contained=False, policy=POLICY_RIGHTMOST,
                 want=WANT_TEXT | WANT_NUMERIC, stats=True, copy=True):
        """rb_trim_paf: query-overlapping records cut at their best split point (paf.rs:210-305, trim_overlap.rs:36-86); one row
        per record, ordered by query name."""
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_trim_paf(self.h, C.byref(recs.c), int(match_score), int(diff_score), int(indel_score), int(bool(remove_contained)),
                                         policy, want, C.byref(out), C.byref(st) if stats else None))
        res = self._collect_lift(out, st if stats else None, want) if copy else dict(n_out=int(out.n_out), paf_nbytes=int(out.paf_nbytes), n_pairs=int(out.n_pairs))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    # rb trim-paf in steps (multi-GPU form: the ranks OR their `waiting` flags after every round, see rbcuda.h)
    def trim_paf_begin(self, recs: Records, match_score=1, diff_score=1, indel_score=1, policy=POLICY_RIGHTMOST):
        self._check(self.lib.rb_trim_paf_begin(self.h, C.byref(recs.c), int(match_score), int(diff_score), int(indel_score), policy))

    def trim_paf_round(self) -> bool:
        w = C.c_int()
        self._check(self.lib.rb_trim_paf_round(self.h, C.byref(w)))
        return bool(w.value)

    def trim_paf_end(self, remove_contained=False, want=WANT_TEXT | WANT_NUMERIC, stats=True):
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_trim_paf_end(self.h, int(bool(remove_contained)), want, C.byref(out), C.byref(st) if stats else None))
        res = self._collect_lift(out, st if stats else None, want)
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def inflate_bgzf(self, data: bytes) -> bytes:
        """rb_inflate_bgzf: the blocks of a BGZF file (myio.rs:41-64) inflated on the device, CRC-32 / ISIZE verified."""
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.rb_inflate_bgzf(self.h, data, len(data), C.byref(p), C.byref(n)))
        out = C.string_at(p.value, n.value) if n.value else b""
        self.lib.rb_free_text(self.h, p)
        return out

    def invert(self, recs: Records, want=WANT_TEXT | WANT_NUMERIC, copy=True):
        """rb_invert: every record with query and target swapped (paf.rs:1050-1094), rows in file order."""
        out = RbLiftOut()
        self._check(self.lib.rb_invert(self.h, C.byref(recs.c), want, C.byref(out)))
        res = self._collect_lift(out, None, want) if copy else dict(n_out=int(out.n_out), paf_nbytes=int(out.paf_nbytes), n_pairs=int(out.n_pairs))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        return res

    def stats(self, recs: Records, copy=True):
        st = RbStatsOut()
        self._check(self.lib.rb_stats(self.h, C.byref(recs.c), C.byref(st)))
        res = self._collect_stats(st) if copy else dict(n=int(st.n))
        self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def _collect_stats(self, st):
        n = int(st.n)
        return dict(n=n, equal=_np(st.equal, n, np.uint32), diff=_np(st.diff, n, np.uint32), ins=_np(st.ins, n, np.uint32),
                    **{"del": _np(st.del_, n, np.uint32)}, ins_events=_np(st.ins_events, n, np.uint32),
                    del_events=_np(st.del_events, n, np.uint32), matches=_np(st.matches, n, np.uint32),
                    id_by_matches=_np(st.id_by_matches, n, np.float32), id_by_events=_np(st.id_by_events, n, np.float32),
                    id_by_all=_np(st.id_by_all, n, np.float32))

    def _collect_lift(self, out, st, want):
        n = int(out.n_out)
        res = dict(n_out=n, n_pairs=int(out.n_pairs), paf_nbytes=int(out.paf_nbytes))
        if want & WANT_TEXT:
            nb = int(out.paf_nbytes)  # (ctypes.string_at takes a C int: texts of 2 GiB and more go through a buffer view)
            addr = C.cast(out.paf_text, C.c_void_p).value
            res["paf_text"] = bytes(memoryview((C.c_ubyte * nb).from_address(addr))) if nb else b""
            res["line_off"] = _np(out.line_off, n + 1, np.uint64)
        if want & WANT_NUMERIC:
            for k in ("q_st", "q_en", "t_st", "t_en", "nmatch", "aln_len"):
                res[k] = _np(getattr(out, k), n, np.uint64)
            res["rec_idx"], res["win_idx"] = _np(out.rec_idx, n, np.uint32), _np(out.win_idx, n, np.uint32)
        if st is not None:
            res["stats"] = self._collect_stats(st)
        return res

    def liftover_text(self, paf: bytes, bed: bytes, policy=POLICY_RIGHTMOST, want=WANT_TEXT | WANT_NUMERIC, stats=True):
        """rb_liftover_text: PAF and BED bytes (text or BGZF) in, the rows of rb_liftover out; on a multi-device context every device
        parses and lifts its share of the PAF.  The dict of liftover() plus "paf_info" and "bed_info"."""
        out, st, pi, bi = RbLiftOut(), RbStatsOut(), RbPafInfo(), RbBedInfo()
        self._check(self.lib.rb_liftover_text(self.h, paf, len(paf), bed, len(bed), policy, want, C.byref(out), C.byref(st) if stats else None,
                                              C.byref(pi), C.byref(bi)))
        res = self._collect_lift(out, st if stats else None, want | (WANT_TEXT if want & WANT_STATS_TEXT else 0))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        res["paf_info"] = _paf_info(pi)
        res["bed_info"] = {k: int(getattr(bi, k)) for k, _ in RbBedInfo._fields_}
        return res

    def stats_text(self, paf: bytes, qbed=False, want=WANT_STATS_TEXT, stats=True):
        """rb_stats_text: PAF bytes (text or BGZF) in, the rows of `rb stats --paf [--qbed]` (without the header line) out, one per
        record in file order; on a multi-device context every device parses and formats its share.  The dict of liftover_text()
        without "bed_info"; want=0 returns the counters only."""
        out, st, pi = RbLiftOut(), RbStatsOut(), RbPafInfo()
        self._check(self.lib.rb_stats_text(self.h, paf, len(paf), int(bool(qbed)), want, C.byref(out), C.byref(st) if stats else None, C.byref(pi)))
        res = self._collect_lift(out, st if stats else None, WANT_TEXT if want & WANT_STATS_TEXT else 0)
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        res["paf_info"] = _paf_info(pi)
        return res

    # ---- resident batches ----
    def upload(self, recs: Records, wins: Windows = None):
        st = C.c_int(0)
        b = self.lib.rb_batch_upload(self.h, C.byref(recs.c), C.byref(wins.c) if wins is not None else None, C.byref(st))
        if not b:
            raise RbError(st.value, self.lib.rb_last_error(self.h).decode())
        return b

    def upload_paf(self, data: bytes):
        """rb_batch_upload_paf: PAF text (or BGZF bytes) parsed on the device into a resident batch without windows.
        Returns (batch, info); info["names"] is the batch's name table (list of bytes, ids by first appearance)."""
        st, info = C.c_int(0), RbPafInfo()
        b = self.lib.rb_batch_upload_paf(self.h, data, len(data), C.byref(info), C.byref(st))
        if not b:
            raise RbError(st.value, self.lib.rb_last_error(self.h).decode())
        nn = int(info.n_names)
        off = _np(info.names_off, nn + 1, np.uint64)
        blob = C.string_at(info.names, int(off[-1])) if nn and int(off[-1]) else b""
        names = [blob[int(off[i]):int(off[i + 1])] for i in range(nn)]
        return b, dict(names=names, n_rec=int(info.n_rec), n_lines=int(info.n_lines), skipped=int(info.skipped),
                       text_bytes=int(info.text_bytes), cigar_bytes=int(info.cigar_bytes))

    def batch_set_windows(self, b, wins):
        """rb_batch_set_windows: windows (t_id = ids of the batch's name table) for a batch uploaded without them."""
        self._check(self.lib.rb_batch_set_windows(self.h, b, C.byref(wins.c) if wins is not None else None))

    def batch_set_windows_bed(self, b, data: bytes) -> dict:
        """rb_batch_set_windows_bed: BED text (or BGZF bytes) parsed on the device into the batch's windows; returns rb_bed_info."""
        info = RbBedInfo()
        self._check(self.lib.rb_batch_set_windows_bed(self.h, b, data, len(data), C.byref(info)))
        return {k: int(getattr(info, k)) for k, _ in RbBedInfo._fields_}

    def batch_windows(self, b) -> dict:
        """rb_batch_windows: the batch's windows as numpy arrays in the rb_windows layout; ids_off / ids are None for default ids."""
        w = RbWindows()
        self._check(self.lib.rb_batch_windows(self.h, b, C.byref(w)))
        n = int(w.n_win)
        res = dict(n_win=n, t_id=_np(w.t_id, n, np.uint32), st=_np(w.st, n, np.uint64), en=_np(w.en, n, np.uint64),
                   bed_row=_np(w.bed_row, n, np.uint32), ids_off=None, ids=None)
        if w.ids_off:
            res["ids_off"] = _np(w.ids_off, n + 1, np.uint64)
            nb = int(res["ids_off"][-1])
            res["ids"] = C.string_at(w.ids, nb) if nb else b""
        return res

    def batch_records(self, b, with_cigar=True) -> dict:
        """rb_batch_records: the batch's records as numpy arrays named like Records' fields (names: list of bytes)."""
        r = RbRecords()
        self._check(self.lib.rb_batch_records(self.h, b, int(with_cigar), C.byref(r)))
        n, nn = int(r.n_rec), int(r.n_names)
        names_off = _np(r.names_off, nn + 1, np.uint64)
        blob = C.string_at(r.names, int(names_off[-1])) if nn and int(names_off[-1]) else b""
        res = dict(n_rec=n, cigar_off=_np(r.cigar_off, n + 1, np.uint64), strand=_np(r.strand, n, np.uint8),
                   q_id=_np(r.q_id, n, np.uint32), t_id=_np(r.t_id, n, np.uint32),
                   names=[blob[int(names_off[i]):int(names_off[i + 1])] for i in range(nn)])
        for k in ("q_len", "q_st", "q_en", "t_len", "t_st", "t_en", "mapq"):
            res[k] = _np(getattr(r, k), n, np.uint64)
        if with_cigar:
            nb = int(r.cigar_nbytes)
            addr = C.cast(r.cigar, C.c_void_p).value  # (a buffer view: string_at takes a C int)
            res["cigar"] = np.frombuffer((C.c_ubyte * nb).from_address(addr), dtype=np.uint8).copy() if nb else np.zeros(0, np.uint8)
        return res

    def batch_liftover(self, b, policy=POLICY_RIGHTMOST, with_stats=True, want=WANT_TEXT | WANT_NUMERIC):
        s = RbSummary()
        self._check(self.lib.rb_batch_liftover(self.h, b, policy, want, int(with_stats), C.byref(s)))
        return dict(n_ops=int(s.n_ops), n_pairs=int(s.n_pairs), n_out=int(s.n_out), out_bytes=int(s.out_bytes), cigar_bytes=int(s.cigar_bytes))

    def batch_stats(self, b):
        s = RbSummary()
        self._check(self.lib.rb_batch_stats(self.h, b, C.byref(s)))
        return dict(n_ops=int(s.n_ops), cigar_bytes=int(s.cigar_bytes))

    def batch_download_lift(self, b, want=WANT_TEXT | WANT_NUMERIC, stats=True, copy=True):
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_batch_download_lift(self.h, b, want, C.byref(out), C.byref(st) if stats else None))
        res = self._collect_lift(out, st if stats else None, want) if copy else dict(n_out=int(out.n_out), paf_nbytes=int(out.paf_nbytes))
        self.lib.rb_free_lift_out(self.h, C.byref(out))
        if stats:
            self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def batch_download_lift_view(self, b, want=WANT_TEXT | WANT_NUMERIC, stats=True):
        """rb_batch_download_lift without copying: (views, release) as liftover_view returns them."""
        out, st = RbLiftOut(), RbStatsOut()
        self._check(self.lib.rb_batch_download_lift(self.h, b, want, C.byref(out), C.byref(st) if stats else None))
        return self._lift_views(out, st, want, stats)

    def batch_download_stats(self, b):
        st = RbStatsOut()
        self._check(self.lib.rb_batch_download_stats(self.h, b, C.byref(st)))
        res = self._collect_stats(st)
        self.lib.rb_free_stats_out(self.h, C.byref(st))
        return res

    def batch_free(self, b):
        self.lib.rb_batch_free(self.h, b)
