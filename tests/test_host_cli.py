"""CPU tests of the host side: the C-ABI library loads and exports every symbol the header
declares, the tools reject bad command lines like the reference's yaggo parsers (message + exit 1),
and the product fails loudly -- no CPU fallback -- when there is no CUDA device."""
import ctypes
import os

import numpy as np
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "pacbio_b200", "libmegareads_b200.so")
CMR = os.path.join(ROOT, "pacbio_b200", "bin", "create_mega_reads")
JFA = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
LPG = os.path.join(ROOT, "pacbio_b200", "bin", "longest_path_overlap_graph2")
MRG = os.path.join(ROOT, "pacbio_b200", "bin", "merge_coords")
REF_MRG = os.path.join(ROOT, "oracle", "_ref", "merge_coords")
GOLD = os.path.join(ROOT, "tests", "golden", "aligner_output")


@pytest.fixture(scope="module", autouse=True)
def built():
    if not all(os.path.exists(p) for p in (LIB, CMR, JFA, LPG, MRG)):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "pacbio_b200", "csrc"), "all"], stdout=subprocess.DEVNULL)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mega_reads_b200.h")).read()
    declared = set(re.findall(r"\b(mr_[a-z_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(LIB)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing


def test_inputs_checksum_tracks_every_input():
    """mr_inputs_checksum (host code, no device): what decides whether a saved index may be reused."""
    import numpy as np
    import pacbio_b200.api as api
    L = api.lib()
    rng = np.random.default_rng(3)
    n, nseq = 1000, 4
    text = rng.integers(0, 2 ** 63, size=(n + 31) // 32, dtype=np.uint64)
    starts = np.array([0, 200, 500, 800, n], dtype=np.uint64)
    ids = np.arange(9, dtype=np.uint32)
    off = np.array([0, 2, 4, 7, 9], dtype=np.uint64)
    ulen = np.array([60, 70, 80, 90, 100, 110, 120, 130, 140], dtype=np.int32)

    def h(text=text, n=n, starts=starts, ids=ids, off=off, ulen=ulen, m=13, k=15, with_unitigs=True):
        p = lambda a, t: a.ctypes.data_as(t)
        if with_unitigs:
            return L.mr_inputs_checksum(p(text, api.u64p), n, p(starts, api.u64p), nseq, p(ids, api.u32p), p(off, api.u64p),
                                        p(ulen, api.i32p), len(ulen), m, k)
        return L.mr_inputs_checksum(p(text, api.u64p), n, p(starts, api.u64p), nseq, None, None, None, 0, m, k)

    base = h()
    assert base == h() and base != 0
    t2 = text.copy(); t2[5] ^= 1 << 20
    s2 = starts.copy(); s2[2] += 1
    i2 = ids.copy(); i2[3] ^= 1
    u2 = ulen.copy(); u2[0] += 1
    others = [h(text=t2), h(starts=s2), h(ids=i2), h(ulen=u2), h(m=12), h(k=16), h(with_unitigs=False)]
    assert len(set(others + [base])) == len(others) + 1
    # bits of the last word past base n are padding, not input (n = 1000: 8 bases, 16 bits, in the last word)
    t3 = text.copy(); t3[-1] ^= np.uint64(1) << np.uint64(40)
    assert h(text=t3) == base


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="checks the no-device behaviour")
def test_no_cpu_fallback_without_a_device():
    import pacbio_b200 as pb
    with pytest.raises(pb.MrError, match="no CUDA device"):
        pb.Context(0)
    r = subprocess.run([CMR, "-s", "10k", "-m", "17", "-k", "65", "-l", os.path.join(GOLD, "test_unitigs_lengths"),
                        "-r", os.path.join(GOLD, "test_super_reads.fa"), "-p", os.path.join(GOLD, "test_pacbio.fa")],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1
    assert b"no CUDA device" in r.stderr and r.stdout == b""


@pytest.mark.parametrize("args,msg", [
    (["-m", "17", "-k", "65"], b"[-s, --size=uint64] required switch"),
    (["-s", "10k", "-k", "65"], b"[-m, --mer=uint32] required switch"),
    (["-s", "10k", "-m", "17"], b"[-k, --k-mer=uint32] required switch"),
    (["-s", "10k", "-m", "17", "-k", "65", "-l", "a", "-u", "b"], b"mutually exclusive"),
    (["-s", "10x", "-m", "17", "-k", "65"], b"Invalid uint64"),
    (["-s", "10k", "-m", "17", "-k", "65", "-T", "bogus"], b"Invalid enum"),
    (["-s", "10k", "-m", "17", "-k", "65", "extra"], b"Requires exactly 0 argument"),
])
def test_create_mega_reads_rejects_bad_command_lines(args, msg):
    r = subprocess.run([CMR] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1
    assert msg in r.stderr


@pytest.mark.parametrize("args,msg", [
    (["coords.txt"], b"[-k, --k-mer=uint32] required switch"),
    (["-k", "41"], b"Requires exactly 1 argument"),
    (["-k", "41", "coords.txt"], b"One of --unitigs-lengths or --unitigs-sequences is required"),
    (["-k", "41", "-l", "a", "-u", "b", "coords.txt"], b"mutually exclusive"),
    (["-k", "41", "-l", "a", "-T", "weighted", "coords.txt"], b"Invalid enum"),
])
def test_longest_path_rejects_bad_command_lines(args, msg):
    """longest_path_overlap_graph2_cmdline.yaggo + longest_path_overlap_graph2.cc:71-72"""
    r = subprocess.run([LPG] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and msg in r.stderr and r.stdout == b""


def test_merge_coords(tmp_path):
    """merge_coords.cc:11-84: per read, the rows of every input in input order; same reads in the same order required."""
    g = os.path.join(ROOT, "tests", "golden")
    a = os.path.join(g, "synth_g1.coords.txt")
    # a second file over the same reads: every other row of the first, reads without rows kept as ">0 name"
    b = str(tmp_path / "b.txt")
    with open(b, "w") as f:
        rec = []
        for line in open(a).read().splitlines() + [">"]:
            if line.startswith(">"):
                if rec:
                    keep = rec[1::2]
                    f.write(">%d %s\n" % (len(keep), rec[0].split(" ", 1)[1]))
                    f.write("".join(l + "\n" for l in keep))
                rec = [line]
            else:
                rec.append(line)
    out = subprocess.run([MRG, a, b, a], stdout=subprocess.PIPE, check=True).stdout.decode().splitlines()
    na = {l.split(" ", 1)[1]: int(l[1:].split()[0]) for l in open(a) if l.startswith(">")}
    nb = {l.split(" ", 1)[1].strip(): int(l[1:].split()[0]) for l in open(b) if l.startswith(">")}
    heads = [l for l in out if l.startswith(">")]
    assert len(heads) == len(na)
    for h in heads:
        name = h.split(" ", 1)[1]
        assert int(h[1:].split()[0]) == 2 * na[name + "\n"] + nb[name]
    assert len(out) == len(heads) + 2 * sum(na.values()) + sum(nb.values())
    if os.path.exists(REF_MRG):                     # the compiled reference, when it is there
        want = subprocess.run([REF_MRG, a, b, a], stdout=subprocess.PIPE, check=True).stdout.decode().splitlines()
        assert out == want
    # gzip-compressed inputs (the reference reads its inputs through zstr, merge_coords.cc:38-43), mixed with plain ones
    import gzip
    bz = str(tmp_path / "b.txt.gz")
    with gzip.open(bz, "wb") as f:
        f.write(open(b, "rb").read())
    az = str(tmp_path / "a.coords.gz")
    with gzip.open(az, "wb") as f:
        f.write(open(a, "rb").read())
    assert subprocess.run([MRG, az, bz, a], stdout=subprocess.PIPE, check=True).stdout.decode().splitlines() == out
    if os.path.exists(REF_MRG):
        assert subprocess.run([REF_MRG, az, bz, a], stdout=subprocess.PIPE, check=True).stdout.decode().splitlines() == out
    # one input: copied; none: empty; -o writes the file
    assert subprocess.run([MRG, a], stdout=subprocess.PIPE, check=True).stdout == open(a, "rb").read()
    assert subprocess.run([MRG], stdout=subprocess.PIPE, check=True).stdout == b""
    o = str(tmp_path / "o.txt")
    subprocess.run([MRG, "-o", o, a, b], check=True)
    assert open(o).read().count(">") == len(na)
    # different reads / different order: error, exit 1
    other = os.path.join(g, "synth_g2.coords.txt")
    r = subprocess.run([MRG, a, other], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and (b"Invalid order of query sequence" in r.stderr or b"prematurely" in r.stderr)
    r = subprocess.run([MRG, a, str(tmp_path / "missing")], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"Error opening coords file" in r.stderr


def test_jf_aligner_needs_an_output():
    r = subprocess.run([JFA, "-s", "10k", "-m", "17"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"No output file given" in r.stderr


def test_missing_input_file_is_an_error():
    r = subprocess.run([CMR, "-s", "10k", "-m", "17", "-k", "65", "-l", "/nonexistent/lengths", "-r", "x", "-p", "y"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert r.returncode == 1 and b"Failed to open unitig lengths" in r.stderr


def test_help_exits_zero():
    for tool in (CMR, JFA):
        r = subprocess.run([tool, "--help"], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert r.returncode == 0 and b"Usage" in r.stdout


def test_host_parsers_match_oracle_inputs(tmp_path):
    """numpy packer used by tests/bench == the layout the reference packs (compact_dna.hpp:109-136)."""
    import numpy as np
    import pacbio_b200.api as api
    sr = api.SuperReads(os.path.join(GOLD, "test_super_reads.fa"))
    assert sr.names == ["1R_3F", "5F_4R_2F", "7R_2F"]
    assert sr.n == 9468 and sr.starts.tolist() == [0, 3668, 6668, 9468]
    assert sr.paths[1] == [(5 << 1), (4 << 1) | 1, (2 << 1)]
    assert sr.row_name(1, True) == "2R_4F_5R"
    # base i lives at bits 2*(i%32) of word i//32
    seq = "".join(l.strip() for l in open(os.path.join(GOLD, "test_super_reads.fa")) if not l.startswith(">"))
    for i in (0, 1, 31, 32, 33, 5000, 9467):
        assert (int(sr.text2bit[i // 32]) >> (2 * (i % 32))) & 3 == "ACGT".index(seq[i])
    assert api.parse_sr_name("12F_7R") == [24, 15] and api.parse_sr_name("xF_7R") == []


def test_bench_workload_shapes(tmp_path, monkeypatch):
    """bench.py's two workload shapes (configs[1] by default, --config human for configs[3]) generate their
    inputs with the parameters they name; scaled down here through --genome / --coverage."""
    import argparse
    import sys
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("MR_BENCH_DIR", str(tmp_path))
    monkeypatch.delenv("RANK", raising=False)
    a = argparse.Namespace(gpus=1, genome=60000, coverage=1.0, config="human", batch_bases=1 << 20)
    w, files = bench.data_files(a)
    assert (w["mer"], w["read_len"], w["repeat_frac"], w["sr_cov"]) == (17, 15000, 0.2, 1.4)
    assert all(os.path.exists(files[k]) for k in ("sr", "reads", "unitigs", "unitigs_len"))
    assert files["info"]["superread_bases"] > 60000 and files["info"]["reads"] >= 3
    assert "configs[3]" in bench.config_dict(a, w)["workload"]
    b = argparse.Namespace(gpus=1, genome=60000, coverage=1.0, config="yeast", batch_bases=1 << 20)
    w2, files2 = bench.data_files(b)
    assert (w2["mer"], w2["read_len"]) == (15, 10000) and files2["prefix"] != files["prefix"]
    assert "configs[1]" in bench.config_dict(b, w2)["workload"]


def test_bench_output_dump(tmp_path, monkeypatch):
    """bench.py --dump-outputs (bench.OutputDump) on results of two batches built here: the rows and info lists of a
    seeded sample of the reads, in read order, as float64; the same files from run to run; every result freed; fewer
    reads (the first drawn) when the rows would pass the size budget."""
    import ctypes as C
    import pacbio_b200.api as api
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(8)
    nreads, cut = 200, 120
    rows_of = rng.integers(0, 6, size=nreads)
    keep_alive, batches = [], []
    for first, nr in ((0, cut), (cut, nreads - cut)):
        cnt = rows_of[first:first + nr]
        n = int(cnt.sum())
        v = api.ResultView()
        v.nreads, v.ncoords = nr, n
        arrays = {"read_coords": np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)}
        for f, t in api.ResultView._fields_:
            if f in bench.DUMP_FIELDS and f not in ("info_len", "lstart", "lprev", "lpath", "lunitigs", "component"):
                dt = {api.u8p: np.uint8, api.i32p: np.int32, api.u32p: np.uint32, api.f64p: np.float64}[t]
                arrays[f] = (rng.integers(0, 250, size=n) + (rng.random(n) if dt is np.float64 else 0)).astype(dt)
        arrays["info_len"] = rng.integers(0, 4, size=n).astype(np.uint32)
        arrays["info_off"] = (np.cumsum(arrays["info_len"]) - arrays["info_len"])[rng.permutation(n)].astype(np.uint64)
        tot = int(arrays["info_len"].sum()) + 1
        arrays["kmers_info"], arrays["bases_info"] = rng.integers(-9, 99, size=tot).astype(np.int32), rng.integers(0, 99, size=tot).astype(np.int32)
        for f, a in arrays.items():
            setattr(v, f, a.ctypes.data_as(dict(api.ResultView._fields_)[f]))
        keep_alive.append(arrays)
        batches.append((first, v))

    def run(path):
        freed = []
        d = bench.OutputDump(nreads, view=lambda h: h, free=freed.append)
        for first, v in reversed(batches):                  # batches may come back in any order
            d.put(first, v)
        d.write(str(path))
        assert sorted(map(id, freed)) == sorted(id(v) for _, v in batches)
        return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}

    got = run(tmp_path / "a")
    assert all(a.dtype == np.float64 for a in got.values())
    assert "lpath" not in got                                # graph fields: not computed, not written
    reads = got["read_index"].astype(np.int64)
    assert len(reads) == nreads // 8 and np.all(np.diff(reads) > 0)
    assert np.array_equal(got["read_rows"], rows_of[reads])
    want = {k: [] for k in got if k not in ("read_index", "read_rows")}
    for r in reads:
        a, first = (keep_alive[0], 0) if r < cut else (keep_alive[1], cut)
        rc = a["read_coords"].astype(np.int64)
        for row in range(rc[r - first], rc[r - first + 1]):
            for k in want:
                if k in ("kmers_info", "bases_info"):
                    o, n = int(a["info_off"][row]), int(a["info_len"][row])
                    want[k].extend(a[k][o:o + n].tolist())
                else:
                    want[k].append(a[k][row])
    for k, w in want.items():
        assert np.array_equal(got[k], np.array(w, dtype=np.float64)), k
    again = run(tmp_path / "b")
    assert all(np.array_equal(got[k], again[k]) for k in got)
    # a budget for about half of the sample: the reads drawn first stay, with all their rows
    row_bytes = 8 * (sum(1 for k in got if k in bench.DUMP_FIELDS) + 2 * got["info_len"].mean())
    monkeypatch.setattr(bench, "DUMP_BYTES", int(row_bytes * got["read_rows"].sum() / 2))
    small = run(tmp_path / "c")
    assert 0 < len(small["read_index"]) < len(reads)
    draw = np.random.default_rng(0).permutation(nreads)
    kept = set(small["read_index"].astype(int).tolist())
    assert max(draw[list(kept)]) < min(draw[[r for r in reads if r not in kept]])
    assert len(small["rs"]) == small["read_rows"].sum()


def test_fixed_point_formatter_prints_what_printf_prints():
    """The mega-read lines carry "%.2f" / "%.4f" doubles (overlap_graph.cc:285-290); the host formatter prints
    them with its own exact routine instead of glibc's (13x faster): same strings on 2e6 operands."""
    import ctypes as C
    H = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    H.mrh_selftest_fixed_format.restype = C.c_uint64
    H.mrh_selftest_fixed_format.argtypes = [C.c_uint64, C.c_uint64]
    assert H.mrh_selftest_fixed_format(2_000_000, 7) == 0


def test_pack_reads_layout():
    """mr_pack_reads: base g at bits 2 (g % 32) of code word g / 32 (compact_dna.hpp:102-136 layout, A0 C1 G2 T3),
    bit g % 64 of mask word g / 64 set for every character outside ACGTacgt (they break k-mers, jf_aligner.hpp:41-52)."""
    import pacbio_b200.api as api
    rng = np.random.default_rng(3)
    for n in (0, 1, 31, 32, 33, 63, 64, 65, 1000, 4097):
        seq = rng.choice(np.frombuffer(b"ACGTacgtNnRY-", dtype=np.uint8), size=n)
        codes, nmask = api.pack_reads(seq)
        assert len(codes) >= (n + 31) // 32 + 4 and len(nmask) >= (n + 63) // 64 + 4
        want = {ord("A"): 0, ord("a"): 0, ord("C"): 1, ord("c"): 1, ord("G"): 2, ord("g"): 2, ord("T"): 3, ord("t"): 3}
        for g in range(n):
            bad = int(nmask[g // 64] >> np.uint64(g % 64)) & 1
            code = int(codes[g // 32] >> np.uint64(2 * (g % 32))) & 3
            if int(seq[g]) in want:
                assert bad == 0 and code == want[int(seq[g])]
            else:
                assert bad == 1 and code == 0
        # nothing set past the last base
        for g in range(n, min(len(nmask) * 64, len(codes) * 32, n + 200)):
            assert (int(nmask[g // 64]) >> (g % 64)) & 1 == 0 and (int(codes[g // 32]) >> (2 * (g % 32))) & 3 == 0


def test_pack_reads_vector_and_portable_forms_agree():
    """The AVX2 packer (32 characters per step) and the byte-at-a-time one (MR_PACK_SCALAR=1) give the same words,
    also when a batch is packed in disjoint word ranges by several threads (mr_pack_reads_range)."""
    import hashlib
    import subprocess
    prog = ("import numpy as np, hashlib, ctypes as C, pacbio_b200.api as api\n"
            "rng = np.random.default_rng(11)\n"
            "seq = rng.choice(np.frombuffer(b'ACGTACGTACGTacgtNnRY-*', dtype=np.uint8), size=1000003)\n"
            "codes, nmask = api.pack_reads(seq)\n"
            "L = api.lib()\n"
            "c2, m2 = np.full(len(codes), 7, np.uint64), np.full(len(nmask), 7, np.uint64)\n"
            "L.mr_pack_reads_range.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]\n"
            "cuts = [0, 1, 17, 5000, 5001, 15000, len(nmask)]\n"
            "for a, b in zip(cuts, cuts[1:]):\n"
            "    assert L.mr_pack_reads_range(seq.ctypes.data, len(seq), a, b - a, c2.ctypes.data, m2.ctypes.data) == 0\n"
            "assert np.array_equal(codes, c2) and np.array_equal(nmask, m2)\n"
            "print(hashlib.sha256(codes.tobytes() + nmask.tobytes()).hexdigest())\n")
    outs = []
    for env in ({}, {"MR_PACK_SCALAR": "1"}):
        r = subprocess.run([sys.executable, "-c", prog], env=dict(os.environ, PYTHONPATH=ROOT, **env), capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-2000:]
        outs.append(r.stdout.strip())
    assert outs[0] == outs[1] and len(outs[0]) == 64


def _fnv(h, data):
    for x in data:
        h = ((h ^ x) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def test_read_stream_parses_fasta_fastq_files_and_pipes(tmp_path):
    """The tools' reader (mapped files scanned in place, pipes in chunks; sequence pieces copied and packed by worker
    threads) against a plain Python parse: FASTA single- and multi-line, FASTQ, CRLF, empty lines, a last line
    without terminator, lower case and N, several files in one stream of batches, small and large batch sizes."""
    import ctypes as C
    import random
    rnd = random.Random(5)
    H = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    H.mrh_selftest_read_stream.argtypes = [C.POINTER(C.c_char_p), C.c_uint, C.c_uint64, C.c_uint, C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]
    recs = [("r%d/x_%d some comment" % (i, i * 7), "".join(rnd.choice("ACGTACGTacgtN") for _ in range(rnd.choice([0, 1, 63, 64, 65, 500, 3000, 12001]))))
            for i in range(60)]
    fa1, fa2, fq = str(tmp_path / "a.fa"), str(tmp_path / "b.fa"), str(tmp_path / "c.fq")
    with open(fa1, "w", newline="") as f:                  # one line per sequence, CRLF on some lines
        for i, (n, s) in enumerate(recs[:20]):
            f.write(">%s%s" % (n, "\r\n" if i % 3 == 0 else "\n"))
            f.write(s + ("\r\n" if i % 3 == 0 else "\n"))
    with open(fa2, "w") as f:                               # 61 columns, empty lines, no final newline
        for n, s in recs[20:40]:
            f.write(">%s\n" % n)
            for i in range(0, len(s), 61):
                f.write(s[i:i + 61] + "\n")
            f.write("\n")
        f.write(">last\nACGTNACGT")
    with open(fq, "w") as f:
        for n, s in recs[40:]:
            f.write("@%s\n" % n)
            half = len(s) // 2
            f.write(s[:half] + "\n" + s[half:] + "\n+\n" + "I" * half + "\n" + "+" * (len(s) - half) + "\n")
    all_recs = recs[:40] + [("last", "ACGTNACGT")] + recs[40:]
    want_bases = "".join(s for _, s in all_recs).encode()
    want_names = "".join(n.split()[0] + "\n" for n, _ in all_recs).encode()
    code = {ord(c): v for c, v in zip("ACGTacgt", [0, 1, 2, 3, 0, 1, 2, 3])}
    h0 = 1469598103934665603
    want = [len(all_recs), len(want_bases), _fnv(h0, want_bases), _fnv(h0, want_names),
            _fnv(h0, bytes(code.get(x, 4) for x in want_bases)), sum(1 for x in want_bases if x not in code)]

    def parse(paths, batch, threads):
        arr = (C.c_char_p * len(paths))(*[p.encode() for p in paths])
        out = (C.c_uint64 * 6)()
        err = C.create_string_buffer(300)
        rc = H.mrh_selftest_read_stream(arr, len(paths), batch, threads, out, err, 300)
        assert rc == 0, err.value
        return list(out)

    for batch, threads in ((1 << 30, 4), (5000, 3), (1, 1), (40000, 8)):
        assert parse([fa1, fa2, fq], batch, threads) == want
    # a mapped FASTA file of several MB: its records are found by all threads at once (read_stream::prescan), each
    # thread starting at the first '>' that begins a line inside its share; one thread takes the serial scanner
    big = str(tmp_path / "big.fa")
    with open(big, "w", newline="") as f:
        for i in range(900):
            s = "".join(rnd.choice("ACGTN") for _ in range(rnd.choice([0, 7, 2000, 9000, 20011])))
            f.write(">big%d with a > sign and\ttabs%s" % (i, "\r\n" if i % 5 == 0 else "\n"))
            cols = rnd.choice([60, 70, 20011])
            for j in range(0, len(s), cols):
                f.write(s[j:j + cols] + ("\r\n" if i % 5 == 0 else "\n"))
            if i % 7 == 0:
                f.write("\n")
    assert os.path.getsize(big) > (4 << 20)
    serial = parse([big], 1 << 21, 1)
    assert serial[0] == 900
    for batch, threads in ((1 << 21, 8), (1 << 30, 5), (30000, 3)):
        assert parse([big, fa2], batch, threads)[:2] == [serial[0] + 21, serial[1] + len("".join(s for _, s in recs[20:40])) + 9]
        assert parse([big], batch, threads) == serial
    # the same bytes through a pipe (stream mode: no mmap, no seek)
    fifo = str(tmp_path / "pipe.fa")
    os.mkfifo(fifo)
    cat = subprocess.Popen("cat %s %s > %s" % (fa1, fa2, fifo), shell=True)
    got = parse([fifo, fq], 7000, 4)
    cat.wait()
    # fa1 + fa2 concatenated: fa1 ends with a newline, so the records are the same
    assert got == want
    bad = str(tmp_path / "bad.txt")
    open(bad, "w").write("not a sequence file\n")
    arr = (C.c_char_p * 1)(bad.encode())
    err = C.create_string_buffer(300)
    assert H.mrh_selftest_read_stream(arr, 1, 1000, 1, (C.c_uint64 * 6)(), err, 300) == -1 and b"Unsupported format" in err.value
