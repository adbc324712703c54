"""ctypes binding of include/mega_reads_b200.h plus numpy helpers to build its inputs.

Mirrors the reference's class seams (SURVEY.md 8b):
    superread_parse(...) -> sequence_psa      ==  Context.index_from_fasta(...) -> Index
    PSA::search                                ==  Index.lookup(mers)
    coarse_aligner::thread::align_sequence_max ==  Context.align(index, reads, params) -> Result

The shared library is REQUIRED: there is no CPU fallback, importing this module without
pacbio_b200/libmegareads_b200.so raises, and creating a Context without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmegareads_b200.so")

u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
u8p = C.POINTER(C.c_uint8)
f64p = C.POINTER(C.c_double)


class MrError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("stretch_factor", C.c_double), ("stretch_constant", C.c_double), ("stretch_cap", C.c_double),
                ("window_size", C.c_uint32), ("forward", C.c_int32), ("max_match", C.c_int32),
                ("max_count", C.c_int32), ("matching_mers", C.c_double), ("matching_bases", C.c_double),
                ("unitigs_k", C.c_uint32), ("overlap_play", C.c_double), ("errors", C.c_double),
                ("bases", C.c_int32), ("run_graph", C.c_int32), ("fine_mer", C.c_uint32)]


class ResultView(C.Structure):
    _fields_ = [("nreads", C.c_uint32), ("ncoords", C.c_uint64), ("read_coords", u64p),
                ("rs", i32p), ("re", i32p), ("qs", i32p), ("qe", i32p), ("nb_mers", i32p),
                ("pb_cons", u32p), ("sr_cons", u32p), ("pb_cover", u32p), ("sr_cover", u32p),
                ("ql", u32p), ("sr", u32p), ("rn", u8p), ("use_bwd", u8p),
                ("stretch", f64p), ("offset", f64p), ("avg_err", f64p),
                ("info_off", u64p), ("info_len", u32p), ("kmers_info", i32p), ("bases_info", i32p),
                ("start_node", u8p), ("end_node", u8p),
                ("lstart", i32p), ("lprev", i32p), ("lpath", i32p), ("lunitigs", i32p), ("component", i32p),
                ("n_kmers_looked_up", C.c_uint64), ("n_tail_entries", C.c_uint64), ("n_hits", C.c_uint64),
                ("n_groups", C.c_uint64), ("n_lists", C.c_uint64), ("n_buckets", C.c_uint64)]


class RecordsParams(C.Structure):
    _fields_ = [("unitigs_k", C.c_uint32), ("overlap_play", C.c_double), ("density", C.c_double),
                ("min_length", C.c_double), ("tiling", C.c_int32), ("trim", C.c_int32)]


class CoordsParams(C.Structure):
    _fields_ = [("compact", C.c_int32), ("zero_match", C.c_int32)]


def records_params(unitigs_k, **kw):
    """The printing options of create_mega_reads (-k, -O, -d, -L, -T as 0 none / 1 greedy / 2 maximal / 3 weighted, --trim)."""
    p = RecordsParams(unitigs_k=unitigs_k, overlap_play=1.3, density=0.029, min_length=100.0, tiling=1, trim=0)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


_lib = None


def lib():
    """Loads the CUDA library; raises if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MrError("pacbio_b200/libmegareads_b200.so is missing: build it with `make -C pacbio_b200/csrc` "
                      "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.mr_context_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.mr_context_destroy.argtypes = [C.c_void_p]
    L.mr_last_error.restype = C.c_char_p
    L.mr_last_error.argtypes = [C.c_void_p]
    L.mr_context_timers.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), f64p, C.c_int]
    L.mr_context_launches.restype = C.c_uint64
    L.mr_context_launches.argtypes = [C.c_void_p]
    L.mr_context_sync.argtypes = [C.c_void_p]
    L.mr_context_stream.restype = C.c_void_p
    L.mr_context_stream.argtypes = [C.c_void_p]
    L.mr_context_keep_taps.argtypes = [C.c_void_p, C.c_int]
    L.mr_index_create.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p, C.c_uint32, u32p, u64p, i32p, C.c_uint32,
                                  C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_index_destroy.argtypes = [C.c_void_p]
    L.mr_index_save.argtypes = [C.c_void_p, C.c_char_p]
    L.mr_index_load.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
    L.mr_index_checksum.restype = C.c_uint64
    L.mr_index_checksum.argtypes = [C.c_void_p]
    L.mr_inputs_checksum.restype = C.c_uint64
    L.mr_inputs_checksum.argtypes = [u64p, C.c_uint64, u64p, C.c_uint32, u32p, u64p, i32p, C.c_uint32, C.c_uint32, C.c_uint32]
    L.mr_selftest_random_gather.restype = C.c_int
    L.mr_selftest_random_gather.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_double)]
    L.mr_index_parts.restype = C.c_uint32
    L.mr_index_parts.argtypes = [C.c_void_p]
    L.mr_index_table_bytes.restype = C.c_uint64
    L.mr_index_table_bytes.argtypes = [C.c_void_p]
    L.mr_index_peek_checksum.argtypes = [C.c_char_p, u64p]
    L.mr_index_sa_size.restype = C.c_uint64
    L.mr_index_sa_size.argtypes = [C.c_void_p]
    L.mr_index_export_sa.argtypes = [C.c_void_p, u64p]
    L.mr_index_export_counts.argtypes = [C.c_void_p, u64p]
    L.mr_lookup_batch.argtypes = [C.c_void_p, u64p, C.c_uint64, u64p, u64p]
    L.mr_lookup_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
    L.mr_params_default.argtypes = [C.POINTER(Params)]
    L.mr_align_batch.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, u64p, C.c_uint32,
                                 C.POINTER(C.c_void_p)]
    L.mr_align_batch_device.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_void_p, u64p,
                                        C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_packed_code_words.restype = C.c_uint64
    L.mr_packed_code_words.argtypes = [C.c_uint64]
    L.mr_packed_mask_words.restype = C.c_uint64
    L.mr_packed_mask_words.argtypes = [C.c_uint64]
    L.mr_pack_reads.argtypes = [C.c_void_p, C.c_uint64, u64p, u64p]
    L.mr_align_batch_packed.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params), u64p, u64p, u64p, C.c_uint32,
                                        C.POINTER(C.c_void_p)]
    L.mr_align_batch_device_packed.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, C.c_void_p, C.c_void_p, u64p,
                                               C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_stage_batch_packed.argtypes = [C.c_void_p, u64p, u64p, u64p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_stage_batch.argtypes = [C.c_void_p, C.c_void_p, u64p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_align_staged.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Params), C.c_void_p, C.POINTER(C.c_void_p)]
    L.mr_staged_free.argtypes = [C.c_void_p]
    L.mr_result_free.argtypes = [C.c_void_p]
    L.mr_result_get.argtypes = [C.c_void_p, C.POINTER(ResultView)]
    L.mr_result_taps.argtypes = [C.c_void_p, u64p, C.POINTER(i64p), u64p, C.POINTER(i32p), u64p, C.POINTER(u32p)]
    L.mr_graph_batch.argtypes = [C.c_void_p, C.POINTER(Params), C.POINTER(ResultView), u32p, u32p, u64p, C.c_uint32, i32p,
                                 C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_unitigs_create.argtypes = [C.c_void_p, C.c_char_p, u64p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_unitigs_destroy.argtypes = [C.c_void_p]
    L.mr_records.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(RecordsParams), C.c_void_p, C.c_char_p, u64p,
                             C.POINTER(C.c_void_p)]
    L.mr_sr_names_create.argtypes = [C.c_void_p, C.c_char_p, u64p, u32p, u64p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.mr_sr_names_destroy.argtypes = [C.c_void_p]
    L.mr_coords_records.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(CoordsParams), C.c_void_p, C.c_char_p, u64p,
                                    C.POINTER(C.c_void_p)]
    L.mr_text_get.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), u64p]
    L.mr_text_free.argtypes = [C.c_void_p]
    _lib = L
    return L


def _p(a, t):
    return a.ctypes.data_as(t)


# -------------------------------------------------------------------------------------------------
# numpy input helpers (test / bench scale; the C++ tools have their own streaming parsers)
# -------------------------------------------------------------------------------------------------
def parse_sr_name(name):
    """(id << 1) | (ori == 'R') list, [] when the name does not parse (super_read_name.cc:74-90)."""
    out = []
    if not name:
        return out
    for piece in name.split("_"):
        digits = ""
        for ch in piece:
            if ch.isdigit():
                digits += ch
            else:
                break
        if not digits:
            return []
        out.append(((int(digits) & 0x7FFFFFFF) << 1) | (1 if piece.endswith("R") else 0))
    return out


def pack_2bit(codes):
    """codes: uint8 array of 0..3 -> uint64 words, base i at bits 2*(i%32) of word i//32."""
    n = len(codes)
    pad = (-n) % 32
    c = np.concatenate([codes, np.zeros(pad, np.uint8)]).astype(np.uint64).reshape(-1, 32)
    shifts = (2 * np.arange(32, dtype=np.uint64))
    return np.bitwise_or.reduce(c << shifts, axis=1)


def load_fasta(path):
    """-> (names, concatenated uint8 sequence bytes, start offsets[n+1]); multi-line records allowed."""
    data = np.fromfile(path, dtype=np.uint8)
    nl = np.flatnonzero(data == 10)
    line_start = np.concatenate([[0], nl + 1])
    line_end = np.concatenate([nl, [len(data)]])
    if line_start[-1] >= len(data):
        line_start, line_end = line_start[:-1], line_end[:-1]
    is_hdr = data[line_start] == ord(">")
    names = [bytes(data[s + 1:e]).decode() for s, e in zip(line_start[is_hdr], line_end[is_hdr])]
    keep = np.ones(len(data), dtype=bool)
    keep[nl] = False
    for s, e in zip(line_start[is_hdr], line_end[is_hdr]):
        keep[s:e] = False
    rec_id = np.cumsum(is_hdr) - 1
    line_len = (line_end - line_start) * (~is_hdr)
    lens = np.bincount(rec_id, weights=line_len, minlength=len(names)).astype(np.uint64)
    starts = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    return names, data[keep], starts


def pack_reads(bases):
    """uint8 characters -> (codes, nmask) as mr_pack_reads lays them out (padding words included)."""
    L = lib()
    bases = np.ascontiguousarray(bases, dtype=np.uint8)
    codes = np.zeros(L.mr_packed_code_words(len(bases)), dtype=np.uint64)
    nmask = np.zeros(L.mr_packed_mask_words(len(bases)), dtype=np.uint64)
    rc = L.mr_pack_reads(bases.ctypes.data_as(C.c_void_p), len(bases), _p(codes, u64p), _p(nmask, u64p))
    if rc != 0:
        raise MrError("mr_pack_reads failed (%d)" % rc)
    return codes, nmask


class SuperReads:
    """What sequence_psa::append_fasta + frag_info hold (superread_parser.cc:12-46, frag_info.hpp:18-35)."""

    def __init__(self, path):
        names, seq, starts = load_fasta(path)
        nonempty = np.diff(starts.astype(np.int64)) > 0
        self.names = [n for n, k in zip(names, nonempty) if k]
        self.starts = np.concatenate([[0], starts[1:][nonempty]]).astype(np.uint64)
        codes = ((seq >> 1) ^ (seq >> 2)) & 3
        self.n = int(len(codes))
        self.text2bit = pack_2bit(codes.astype(np.uint8))
        paths = [parse_sr_name(n) for n in self.names]
        self.unitig_off = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.uint64)
        self.unitig_ids = np.array([x for p in paths for x in p], dtype=np.uint32)
        self.paths = paths

    def row_name(self, sr, bwd):
        p = self.paths[sr]
        if not bwd or not p:
            return self.names[sr]
        return "_".join("%d%s" % (x >> 1, "F" if x & 1 else "R") for x in reversed(p))


class Reads:
    def __init__(self, path=None, names=None, seqs=None):
        if path is not None:
            names, seq, starts = load_fasta(path)
            self.names = [n.split()[0] if n.split() else "" for n in names]
            self.bases, self.starts = np.ascontiguousarray(seq), starts
        else:
            self.names = list(names)
            self.bases = np.frombuffer("".join(seqs).encode(), dtype=np.uint8).copy()
            self.starts = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.uint64)

    @property
    def nreads(self):
        return len(self.names)

    def slice(self, lo, hi):
        r = Reads.__new__(Reads)
        r.names = self.names[lo:hi]
        b0, b1 = int(self.starts[lo]), int(self.starts[hi])
        r.bases = np.ascontiguousarray(self.bases[b0:b1])
        r.starts = (self.starts[lo:hi + 1] - self.starts[lo]).astype(np.uint64)
        return r


# -------------------------------------------------------------------------------------------------
# handles
# -------------------------------------------------------------------------------------------------
class Context:
    def __init__(self, device=0):
        L = lib()
        h = C.c_void_p()
        rc = L.mr_context_create(device, C.byref(h))
        if rc != 0:
            raise MrError("mr_context_create failed (%d): %s" % (rc, L.mr_last_error(None).decode()))
        self.h, self.L = h, L

    def close(self):
        if self.h:
            self.L.mr_context_destroy(self.h)
            self.h = None

    def check(self, rc):
        if rc != 0:
            raise MrError("error %d: %s" % (rc, self.L.mr_last_error(self.h).decode()))

    def timers(self):
        names = (C.c_char_p * 32)()
        secs = (C.c_double * 32)()
        n = self.L.mr_context_timers(self.h, names, secs, 32)
        return {names[i].decode(): secs[i] for i in range(n)}

    def launches(self):
        return int(self.L.mr_context_launches(self.h))

    def sync(self):
        self.check(self.L.mr_context_sync(self.h))

    def stream(self):
        return self.L.mr_context_stream(self.h)

    def keep_taps(self, on=True):
        self.check(self.L.mr_context_keep_taps(self.h, int(on)))

    def index(self, sr, psa_min, k, unitig_len=None):
        return Index(self, sr, psa_min, k, unitig_len)

    def align(self, index, reads, params, keep=False):
        """keep: the Result holds on to the native result (for records()) until its close()."""
        out = C.c_void_p()
        starts = np.ascontiguousarray(reads.starts, dtype=np.uint64)
        self.check(self.L.mr_align_batch(self.h, index.h, C.byref(params), reads.bases.ctypes.data_as(C.c_void_p),
                                         _p(starts, u64p), reads.nreads, C.byref(out)))
        return Result(self, out, keep)

    def graph(self, rows, read_len, path_ids, path_off, unitig_len, params):
        """mr_graph_batch over rows the caller made: `rows` maps every coords column of ResultView (and read_coords,
        kmers_info, bases_info) to a numpy array; path_ids / path_off is the unitig-path table rows["sr"] indexes.
        The Result keeps its native object, so that records() can print it."""
        dt = {u8p: np.uint8, i32p: np.int32, u32p: np.uint32, f64p: np.float64, u64p: np.uint64}
        v = ResultView()
        keep = []
        for name, t in ResultView._fields_:
            if name in rows:
                a = np.ascontiguousarray(rows[name], dtype=dt[t])
                if len(a) == 0:
                    a = np.zeros(1, dtype=dt[t])
                keep.append(a)
                setattr(v, name, _p(a, t))
        v.nreads = len(rows["read_coords"]) - 1
        v.ncoords = int(rows["read_coords"][-1])
        rl = np.ascontiguousarray(read_len, dtype=np.uint32)
        ids = np.ascontiguousarray(path_ids if len(path_ids) else [0], dtype=np.uint32)
        off = np.ascontiguousarray(path_off, dtype=np.uint64)
        ul = np.ascontiguousarray(unitig_len, dtype=np.int32)
        out = C.c_void_p()
        self.check(self.L.mr_graph_batch(self.h, C.byref(params), C.byref(v), _p(rl, u32p), _p(ids, u32p), _p(off, u64p),
                                         len(off) - 1, _p(ul, i32p), len(ul), C.byref(out)))
        return Result(self, out, True)

    def unitigs(self, seq, off):
        """The k-unitig sequences on this context's device (mr_unitigs_create): seq bytes, off[n + 1]."""
        return Unitigs(self, seq, off)

    def records(self, result, names, params, unitigs=None):
        """The create_mega_reads records of `result` (which must be this context's latest, kept with keep=True),
        printed on the device (mr_records); unitigs: Unitigs for the sequence column (-u), None for -l."""
        if result.h is None:
            raise MrError("records() needs a Result that kept its native object (align(..., keep=True) or graph())")
        enc, off = _joined(names)
        t = C.c_void_p()
        self.check(self.L.mr_records(self.h, result.h, C.byref(params), unitigs.h if unitigs is not None else None,
                                     enc, _p(off, u64p), C.byref(t)))
        return self._text(t)

    def sr_names(self, names, path_ids, path_off):
        """The super-reads' names (FASTA headers after '>') and unitig paths (CSR, as SuperReads.unitig_ids /
        unitig_off) on this context's device (mr_sr_names_create), for coords_records()."""
        return SrNames(self, names, path_ids, path_off)

    def coords_records(self, result, names, compact=True, zero_match=False, *, sr_names):
        """The jf_aligner coords lines of `result` (this context's latest, kept with keep=True, or from graph()),
        printed on the device (mr_coords_records): compact is the tool's default format (--compact toggles it off),
        zero_match is -0.  names: the reads' names; sr_names: an SrNames of the table the rows' `sr` indexes."""
        if result.h is None:
            raise MrError("coords_records() needs a Result that kept its native object (align(..., keep=True) or graph())")
        enc, off = _joined(names)
        p = CoordsParams(compact=int(bool(compact)), zero_match=int(bool(zero_match)))
        t = C.c_void_p()
        self.check(self.L.mr_coords_records(self.h, result.h, C.byref(p), sr_names.h, enc, _p(off, u64p), C.byref(t)))
        return self._text(t)

    def _text(self, t):
        try:
            p, n = C.c_void_p(), C.c_uint64()
            self.check(self.L.mr_text_get(t, C.byref(p), C.byref(n)))
            return C.string_at(p, n.value) if n.value else b""
        finally:
            self.L.mr_text_free(t)

    def align_packed(self, index, reads, params):
        """Same as align(), through the packed entry point: the batch is packed on the host (mr_pack_reads) and
        crosses PCIe at 0.375 bytes per base."""
        out = C.c_void_p()
        starts = np.ascontiguousarray(reads.starts, dtype=np.uint64)
        codes, nmask = pack_reads(reads.bases)
        self.check(self.L.mr_align_batch_packed(self.h, index.h, C.byref(params), _p(codes, u64p), _p(nmask, u64p),
                                                _p(starts, u64p), reads.nreads, C.byref(out)))
        return Result(self, out)

    def stage(self, reads):
        """Starts the host -> device copy of a batch (mr_stage_batch); pass the handle to align_staged."""
        h = C.c_void_p()
        starts = np.ascontiguousarray(reads.starts, dtype=np.uint64)
        self.check(self.L.mr_stage_batch(self.h, reads.bases.ctypes.data_as(C.c_void_p), _p(starts, u64p), reads.nreads, C.byref(h)))
        return h

    def align_staged(self, index, staged, params):
        out = C.c_void_p()
        self.check(self.L.mr_align_staged(self.h, index.h, C.byref(params), staged, C.byref(out)))
        return Result(self, out)

    def align_device(self, index, d_bases_ptr, d_starts_ptr, h_starts, nreads, params):
        out = C.c_void_p()
        h_starts = np.ascontiguousarray(h_starts, dtype=np.uint64)
        self.check(self.L.mr_align_batch_device(self.h, index.h, C.byref(params), C.c_void_p(d_bases_ptr),
                                                C.c_void_p(d_starts_ptr), _p(h_starts, u64p), nreads, C.byref(out)))
        return Result(self, out)


def default_params(**kw):
    p = Params()
    lib().mr_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


class Index:
    def __init__(self, ctx, sr, psa_min, k, unitig_len=None, load_from=None):
        """Builds the index of `sr` (a SuperReads) or, with load_from, reads a file written by save()."""
        self.ctx, self.sr, self.m, self.k = ctx, sr, psa_min, k
        h = C.c_void_p()
        if load_from is not None:
            ctx.check(ctx.L.mr_index_load(ctx.h, os.fsencode(load_from), C.byref(h)))
            self.h = h
            return
        if unitig_len is not None:
            ul = np.ascontiguousarray(unitig_len, dtype=np.int32)
            ids = np.ascontiguousarray(sr.unitig_ids, dtype=np.uint32)
            if len(ids) == 0:
                ids = np.zeros(1, np.uint32)
            args = (_p(ids, u32p), _p(sr.unitig_off, u64p), _p(ul, i32p), len(ul))
        else:
            args = (None, None, None, 0)
        ctx.check(ctx.L.mr_index_create(ctx.h, _p(sr.text2bit, u64p), sr.n, _p(sr.starts, u64p), len(sr.names),
                                        *args, psa_min, k, C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            self.ctx.L.mr_index_destroy(self.h)
            self.h = None

    def save(self, path):
        self.ctx.check(self.ctx.L.mr_index_save(self.h, os.fsencode(path)))

    def checksum(self):
        return int(self.ctx.L.mr_index_checksum(self.h))

    def parts(self):
        return int(self.ctx.L.mr_index_parts(self.h))

    def sa(self):
        out = np.empty(self.ctx.L.mr_index_sa_size(self.h), dtype=np.uint64)
        self.ctx.check(self.ctx.L.mr_index_export_sa(self.h, _p(out, u64p)))
        return out

    def counts(self):
        out = np.empty(4 ** self.m + 1, dtype=np.uint64)
        self.ctx.check(self.ctx.L.mr_index_export_counts(self.h, _p(out, u64p)))
        return out

    def lookup(self, mers):
        mers = np.ascontiguousarray(mers, dtype=np.uint64)
        idx = np.empty(len(mers), np.uint64)
        nb = np.empty(len(mers), np.uint64)
        self.ctx.check(self.ctx.L.mr_lookup_batch(self.h, _p(mers, u64p), len(mers), _p(idx, u64p), _p(nb, u64p)))
        return idx, nb


def _joined(names):
    """names (str or bytes) back to back, and their n + 1 offsets"""
    enc = [n.encode() if isinstance(n, str) else bytes(n) for n in names]
    off = np.concatenate([[0], np.cumsum([len(n) for n in enc])]).astype(np.uint64)
    return b"".join(enc), off


def _arr(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


class Unitigs:
    def __init__(self, ctx, seq, off):
        self.ctx = ctx
        off = np.ascontiguousarray(off, dtype=np.uint64)
        h = C.c_void_p()
        ctx.check(ctx.L.mr_unitigs_create(ctx.h, bytes(seq), _p(off, u64p), len(off) - 1, C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            self.ctx.L.mr_unitigs_destroy(self.h)
            self.h = None


class SrNames:
    def __init__(self, ctx, names, path_ids, path_off):
        self.ctx = ctx
        enc, off = _joined(names)
        ids = np.ascontiguousarray(path_ids if len(path_ids) else [0], dtype=np.uint32)
        poff = np.ascontiguousarray(path_off, dtype=np.uint64)
        h = C.c_void_p()
        ctx.check(ctx.L.mr_sr_names_create(ctx.h, enc, _p(off, u64p), _p(ids, u32p), _p(poff, u64p), len(off) - 1, C.byref(h)))
        self.h = h

    def close(self):
        if self.h:
            self.ctx.L.mr_sr_names_destroy(self.h)
            self.h = None


class Result:
    """Copies the pinned result arrays into numpy and frees the native object (with keep: at close())."""

    def __init__(self, ctx, h, keep=False):
        v = ResultView()
        ctx.check(ctx.L.mr_result_get(h, C.byref(v)))
        self.view_struct = None
        n, nr = int(v.ncoords), int(v.nreads)
        self.nreads, self.ncoords = nr, n
        self.read_coords = _arr(v.read_coords, nr + 1, np.uint64)
        for f in ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "sr", "rn",
                  "use_bwd", "stretch", "offset", "avg_err", "info_off", "info_len", "start_node", "end_node",
                  "lstart", "lprev", "lpath", "lunitigs", "component"):
            ptr = getattr(v, f)
            dt = {u8p: np.uint8, i32p: np.int32, u32p: np.uint32, f64p: np.float64, u64p: np.uint64}[type(ptr)]
            setattr(self, f, _arr(ptr, n, dt))
        tot = int((self.info_off + self.info_len).max()) if n and self.info_len.max() > 0 else 0
        self.kmers_info = _arr(v.kmers_info, tot, np.int32)
        self.bases_info = _arr(v.bases_info, tot, np.int32)
        self.n_kmers_looked_up, self.n_hits, self.n_groups = int(v.n_kmers_looked_up), int(v.n_hits), int(v.n_groups)
        ng, no, nl = C.c_uint64(), C.c_uint64(), C.c_uint64()
        pg, po, pl = i64p(), i32p(), u32p()
        ctx.check(ctx.L.mr_result_taps(h, C.byref(ng), C.byref(pg), C.byref(no), C.byref(po), C.byref(nl), C.byref(pl)))
        self.tap_groups = _arr(pg, ng.value * 6, np.int64).reshape(-1, 6)
        self.tap_offsets = _arr(po, no.value * 2, np.int32).reshape(-1, 2)
        self.tap_lis = _arr(pl, nl.value, np.uint32)
        self.ctx, self.h = ctx, None
        if keep:
            self.h = h
        else:
            ctx.L.mr_result_free(h)

    def close(self):
        if self.h:
            self.ctx.L.mr_result_free(self.h)
            self.h = None

    def rows(self, r):
        return range(int(self.read_coords[r]), int(self.read_coords[r + 1]))

    def info(self, row):
        o, l = int(self.info_off[row]), int(self.info_len[row])
        return self.kmers_info[o:o + l], self.bases_info[o:o + l]
