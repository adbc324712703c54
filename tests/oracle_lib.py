"""ctypes bindings for the two CPU checkers (TEST INFRASTRUCTURE, never imported by the product):

* ``Port``  -> oracle/liboracle_port.so : our C++ restatement (always buildable from this repo)
* ``Ref``   -> oracle/_ref/libref_tap.so : the reference's own sources compiled against shims
               (only present when oracle/_ref was built where /root/reference exists; it travels
               to the GPU box as a built file)

Both expose the same stage-level taps, so the same comparison code runs against either.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
PORT_SO = os.path.join(ORACLE_DIR, "liboracle_port.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libref_tap.so")
REF_CMR = os.path.join(ORACLE_DIR, "_ref", "create_mega_reads")
REF_JFA = os.path.join(ORACLE_DIR, "_ref", "jf_aligner")
REF_LP = os.path.join(ORACLE_DIR, "_ref", "longest_path_overlap_graph2")
GEN = os.path.join(ROOT, "pacbio_b200", "tools", "gen_synth")


def build_port():
    if not os.path.exists(PORT_SO):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "port"], stdout=subprocess.DEVNULL)
    return PORT_SO


def have_ref():
    return os.path.exists(REF_SO) and os.path.exists(REF_CMR)


u64p = C.POINTER(C.c_uint64)
i64p = C.POINTER(C.c_int64)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
f64p = C.POINTER(C.c_double)


def _ptr(a, t):
    return a.ctypes.data_as(t)


class _Taps:
    """Uniform wrapper over the op_* / ref_* tap functions."""

    def __init__(self, so, prefix, create_takes_threads):
        self.lib = C.CDLL(so)
        self.p = prefix
        self.create_takes_threads = create_takes_threads
        L = self.lib
        g = lambda n: getattr(L, prefix + n)
        g("index_create").restype = C.c_void_p
        for n in ("index_n", "index_nseq", "index_sa_size", "res_ngroups", "res_noffsets", "res_nlis",
                  "res_ncoords", "res_ninfo"):
            g(n).restype = C.c_uint64
            g(n).argtypes = [C.c_void_p]
        g("index_destroy").argtypes = [C.c_void_p]
        g("index_sa").argtypes = [C.c_void_p, u64p]
        g("index_counts").argtypes = [C.c_void_p, u64p]
        g("index_seq_starts").argtypes = [C.c_void_p, u64p]
        g("index_search").argtypes = [C.c_void_p, u64p, C.c_uint64, u64p, u64p]
        g("lis").restype = C.c_uint32
        g("lis").argtypes = [i32p, C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_uint32, u32p]
        g("index_set_unitigs_lengths").argtypes = [C.c_void_p, i32p, C.c_uint64]
        g("aligner_create").restype = C.c_void_p
        g("aligner_create").argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_uint32, C.c_int, C.c_int,
                                        C.c_int, C.c_double, C.c_double, C.c_uint32]
        g("aligner_destroy").argtypes = [C.c_void_p]
        g("align_read").argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
        g("res_copy").argtypes = [C.c_void_p, i64p, i32p, u32p, i64p, f64p, i64p, i32p, i32p]

    def f(self, name):
        return getattr(self.lib, self.p + name)

    # ---- index -----------------------------------------------------------
    def index_create(self, sr_fasta, m, k, threads=4):
        if self.create_takes_threads:
            self.f("index_create").argtypes = [C.c_char_p, C.c_uint, C.c_uint, C.c_uint]
            h = self.f("index_create")(sr_fasta.encode(), m, k, threads)
        else:
            self.f("index_create").argtypes = [C.c_char_p, C.c_uint, C.c_uint]
            h = self.f("index_create")(sr_fasta.encode(), m, k)
        if not h:
            raise RuntimeError("index_create failed")
        return h

    def index_destroy(self, h):
        self.f("index_destroy")(h)

    def sa(self, h):
        out = np.empty(self.f("index_sa_size")(h), dtype=np.uint64)
        self.f("index_sa")(h, _ptr(out, u64p))
        return out

    def counts(self, h, m):
        out = np.empty(4 ** m + 1, dtype=np.uint64)
        self.f("index_counts")(h, _ptr(out, u64p))
        return out

    def seq_starts(self, h):
        out = np.empty(self.f("index_nseq")(h) + 1, dtype=np.uint64)
        self.f("index_seq_starts")(h, _ptr(out, u64p))
        return out

    def n(self, h):
        return self.f("index_n")(h)

    def search(self, h, mers):
        mers = np.ascontiguousarray(mers, dtype=np.uint64)
        idx = np.empty(len(mers), dtype=np.uint64)
        nb = np.empty(len(mers), dtype=np.uint64)
        self.f("index_search")(h, _ptr(mers, u64p), len(mers), _ptr(idx, u64p), _ptr(nb, u64p))
        return idx, nb

    def search_k(self, h, mers, kk):
        """The fine pass's lookup: patterns of kk <= k bases in the same suffix array."""
        mers = np.ascontiguousarray(mers, dtype=np.uint64)
        idx = np.empty(len(mers), np.uint64)
        nb = np.empty(len(mers), np.uint64)
        f = self.f("index_search_k")
        f.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_uint, u64p, u64p]
        f(h, _ptr(mers, u64p), len(mers), kk, _ptr(idx, u64p), _ptr(nb, u64p))
        return idx, nb

    def lis(self, pairs, a=1.3, b=10.0, cap=10000.0, window=1):
        pairs = np.ascontiguousarray(pairs, dtype=np.int32).reshape(-1, 2)
        out = np.empty(max(1, len(pairs)), dtype=np.uint32)
        n = self.f("lis")(_ptr(pairs, i32p), len(pairs), a, b, cap, window, _ptr(out, u32p))
        return out[:n].copy()

    def set_unitigs_lengths(self, h, lens):
        lens = np.ascontiguousarray(lens, dtype=np.int32)
        self.f("index_set_unitigs_lengths")(h, _ptr(lens, i32p), len(lens))

    # ---- per-read ----------------------------------------------------------
    def aligner_create(self, h, stretch_factor=1.3, stretch_constant=10.0, stretch_cap=10000.0, window_size=1,
                       forward=True, max_match=False, max_count=5000, matching_mers=0.0, matching_bases=0.17,
                       unitigs_k=0):
        return self.f("aligner_create")(h, stretch_factor, stretch_constant, stretch_cap, window_size, int(forward),
                                        int(max_match), max_count, matching_mers, matching_bases, unitigs_k)

    def aligner_destroy(self, a):
        self.f("aligner_destroy")(a)

    def align_read(self, a, seq):
        """Returns dict(groups[n,5], offsets[m,2], lis, cint[c,14], cdbl[c,3], info_off, kinfo, binfo)."""
        if isinstance(seq, str):
            seq = seq.encode()
        rc = self.f("align_read")(a, seq, len(seq))
        if rc != 0:
            raise RuntimeError("align_read failed")
        ng, no, nl = self.f("res_ngroups")(a), self.f("res_noffsets")(a), self.f("res_nlis")(a)
        nc, ni = self.f("res_ncoords")(a), self.f("res_ninfo")(a)
        r = dict(groups=np.empty((ng, 5), np.int64), offsets=np.empty((no, 2), np.int32), lis=np.empty(nl, np.uint32),
                 cint=np.empty((nc, 14), np.int64), cdbl=np.empty((nc, 3), np.float64),
                 info_off=np.empty(nc + 1, np.int64), kinfo=np.empty(ni, np.int32), binfo=np.empty(ni, np.int32))
        self.f("res_copy")(a, _ptr(r["groups"], i64p), _ptr(r["offsets"], i32p), _ptr(r["lis"], u32p),
                           _ptr(r["cint"], i64p), _ptr(r["cdbl"], f64p), _ptr(r["info_off"], i64p),
                           _ptr(r["kinfo"], i32p), _ptr(r["binfo"], i32p))
        return r


class Port(_Taps):
    def __init__(self):
        super().__init__(build_port(), "op_", False)
        L = self.lib
        L.op_kmers_info_trace.argtypes = [C.c_char_p, i32p, C.c_uint32, C.c_uint32, C.c_uint32, i32p, C.c_uint32,
                                          i32p, C.c_uint32]
        L.op_sr_overlap.argtypes = [C.c_char_p, C.c_char_p]
        L.op_run.restype = C.c_int64
        L.op_run.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_uint, C.c_uint,
                             C.c_uint, C.c_uint64, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int,
                             C.c_double, C.c_double, C.c_uint, C.c_double, C.c_double, C.c_double, C.c_double,
                             C.c_int, C.c_int, C.c_int, f64p, f64p]

    def kmers_info_trace(self, name, ul, unitigs_k, k, positions):
        ul = np.ascontiguousarray(ul, dtype=np.int32)
        pos = np.ascontiguousarray(positions, dtype=np.int32)
        out = np.empty(65536, dtype=np.int32)
        w = self.lib.op_kmers_info_trace(name.encode(), _ptr(ul, i32p), len(ul), unitigs_k, k, _ptr(pos, i32p),
                                         len(pos), _ptr(out, i32p), len(out))
        assert w >= 0
        rows, i = [], 0
        while i < w:
            nm = out[i]; mers = out[i + 1:i + 1 + nm].tolist(); i += 1 + nm
            nb = out[i]; bases = out[i + 1:i + 1 + nb].tolist(); i += 1 + nb
            rows.append((mers, bases))
        return rows

    def sr_overlap(self, a, b):
        return self.lib.op_sr_overlap(a.encode(), b.encode())

    def run(self, mode, sr, reads, unitigs, out, mer, k_unitig, unitigs_is_fasta=True, psa_min=13, threads=1,
            max_reads=0, stretch_factor=1.3, stretch_constant=10.0, stretch_cap=10000.0, forward=True,
            max_match=False, max_count=5000, mers_matching=0.0, bases_matching=17.0, overlap_play=1.3, errors=3.0,
            density=0.029, min_length=100.0, bases=False, tiling=1, trim=0, fine_mer=0):
        ti, ta = C.c_double(0), C.c_double(0)
        self.lib.op_set_fine_mer.argtypes = [C.c_uint]
        self.lib.op_set_fine_mer(fine_mer)
        nb = self.lib.op_run(mode, sr.encode(), reads.encode(), (unitigs or "").encode(), int(unitigs_is_fasta),
                             out.encode(), mer, psa_min, threads, max_reads, stretch_factor, stretch_constant,
                             stretch_cap, int(forward), int(max_match), max_count, mers_matching, bases_matching,
                             k_unitig, overlap_play, errors, density, min_length, int(bases), tiling, trim,
                             C.byref(ti), C.byref(ta))
        if nb < 0:
            raise RuntimeError("op_run failed")
        return nb, ti.value, ta.value


class Ref(_Taps):
    def __init__(self):
        if not have_ref():
            raise RuntimeError("oracle/_ref not built")
        super().__init__(REF_SO, "ref_", True)


# ---------------------------------------------------------------------------
# helpers shared by tests
# ---------------------------------------------------------------------------
def gen_synth(prefix, genome, coverage=5, read_len=5000, error=0.15, seed=42, sr_cov=2.0, repeat_frac=0.0,
              unitig_k=41, threads=4, mean_unitig=500):
    if not os.path.exists(GEN):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-pthread", GEN + ".cc", "-o", GEN])
    import json
    out = subprocess.check_output([GEN, "--genome", str(genome), "--coverage", str(coverage), "--read-len",
                                   str(read_len), "--error", str(error), "--seed", str(seed), "--sr-cov", str(sr_cov),
                                   "--repeat-frac", str(repeat_frac), "--unitig-k", str(unitig_k), "--threads",
                                   str(threads), "--mean-unitig", str(mean_unitig), "--prefix", prefix])
    info = json.loads(out)
    info.update(sr=prefix + ".superreads.fa", reads=prefix + ".reads.fa", unitigs=prefix + ".unitigs.fa",
                unitigs_len=prefix + ".unitigs_len.txt")
    return info


def read_fasta(path):
    names, seqs, cur = [], [], []
    with open(path) as f:
        for line in f:
            if line.startswith(">"):
                if names:
                    seqs.append("".join(cur))
                names.append(line[1:].split()[0] if line[1:].split() else "")
                cur = []
            else:
                cur.append(line.strip())
    if names:
        seqs.append("".join(cur))
    return names, seqs


def canon_rows(cint, cdbl, info_off, kinfo, binfo):
    """Coords rows as comparable tuples: integers exact, doubles by their bit pattern (float.hex), each row's
    kmers_info / bases_info slice."""
    rows = []
    for j in range(len(cint)):
        lo, hi = info_off[j], info_off[j + 1]
        rows.append((tuple(int(x) for x in cint[j]), tuple(float(x).hex() for x in cdbl[j]),
                     tuple(kinfo[lo:hi].tolist()), tuple(binfo[lo:hi].tolist())))
    return rows


def oracle_rows(o):
    """canon_rows of one read's result from a checker's align_read."""
    return canon_rows(o["cint"], o["cdbl"], o["info_off"], o["kinfo"], o["binfo"])


def device_rows(res, r, read_len):
    """canon_rows of read r of a pacbio_b200 Result, laid out as the checkers' align_read lays them out
    (cint = rs, re, qs, qe, nb_mers, pb_cons, sr_cons, pb_cover, sr_cover, read length, ql, rn, sr, use_bwd)."""
    rr = list(res.rows(r))
    if not rr:
        return []
    g_int = np.stack([res.rs[rr], res.re[rr], res.qs[rr], res.qe[rr], res.nb_mers[rr], res.pb_cons[rr],
                      res.sr_cons[rr], res.pb_cover[rr], res.sr_cover[rr], np.full(len(rr), read_len), res.ql[rr],
                      res.rn[rr], res.sr[rr], res.use_bwd[rr]], axis=1).astype(np.int64)
    g_dbl = np.stack([res.stretch[rr], res.offset[rr], res.avg_err[rr]], axis=1)
    g_off = np.concatenate([[0], np.cumsum(res.info_len[rr])]).astype(np.int64)
    g_k = np.concatenate([res.info(i)[0] for i in rr])
    g_b = np.concatenate([res.info(i)[1] for i in rr])
    return canon_rows(g_int, g_dbl, g_off, g_k, g_b)


def records(path_or_text, is_text=False):
    """Parse create_mega_reads / compact jf_aligner output into {read header: sorted tuple of lines}."""
    text = path_or_text if is_text else open(path_or_text).read()
    recs, cur = {}, None
    for line in text.splitlines():
        if line.startswith(">"):
            cur = line
            assert cur not in recs, "duplicate record " + cur
            recs[cur] = []
        elif cur is not None:
            recs[cur].append(line)
    return {k: tuple(sorted(v)) for k, v in recs.items()}
