"""jf_aligner coords lines printed on the device (mr_coords_records, Context.coords_records) against the host
formatter (mrh::format_coords, the printer of the --details path) on the same result, byte for byte, in one process;
a round trip through the reference's own coords files; the refusals; and the tool end to end."""
import ctypes as C
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLD = os.path.join(ROOT, "tests", "golden")
JFA = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
PRINTS = [(compact, zero) for compact in (True, False) for zero in (False, True)]


def host_lib():
    H = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    H.mrh_format_coords.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_char_p,
                                    C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                    C.c_char_p, C.c_size_t]
    H.mrh_free.argtypes = [C.c_void_p]
    return H


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def joined(names):
    enc = [n.encode() if isinstance(n, str) else n for n in names]
    return b"".join(enc), np.concatenate([[0], np.cumsum([len(n) for n in enc])]).astype(np.uint64)


def host_coords(H, res, sr_names, path_ids, path_off, names, read_len, compact, zero):
    """What mrh::format_coords prints for the result."""
    srn, sro = joined(sr_names)
    ids = np.ascontiguousarray(path_ids if len(path_ids) else [0], dtype=np.uint32)
    off = np.ascontiguousarray(path_off, dtype=np.uint64)
    rn, ro = joined(names)
    starts = np.concatenate([[0], np.cumsum(np.asarray(read_len, dtype=np.uint64))]).astype(np.uint64)
    out, size, err = C.c_void_p(), C.c_uint64(), C.create_string_buffer(300)
    rc = H.mrh_format_coords(res.h, srn, ptr(sro), ptr(ids), ptr(off), len(off) - 1, rn, ptr(ro), ptr(starts), int(compact),
                             int(zero), C.byref(out), C.byref(size), err, 300)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    text = C.string_at(out, size.value) if size.value else b""
    H.mrh_free(out)
    return text


def compare(ctx, H, res, srn, sr_names, path_ids, path_off, names, read_len, what):
    """compact x -0: device bytes == host bytes.  Returns the texts."""
    texts = {}
    for compact, zero in PRINTS:
        want = host_coords(H, res, sr_names, path_ids, path_off, names, read_len, compact, zero)
        got = ctx.coords_records(res, names, compact, zero, sr_names=srn)
        if got != want:
            a, b = got.split(b"\n"), want.split(b"\n")
            i = next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), min(len(a), len(b)))
            raise AssertionError("%s compact %d -0 %d: line %d differs:\n device %r\n host   %r" % (
                what, compact, zero, i, a[i][:300] if i < len(a) else None, b[i][:300] if i < len(b) else None))
        texts[(compact, zero)] = got
    return texts


def with_edge_super_reads(info, tmp, unknown_id):
    """The fixture's super-reads plus, test_gpu_chain_edges-style, two whose names do not parse (an empty path: their
    backward rows print the header; a piece of the longest super-read in both orientations, so that a read which hits
    it makes a backward row on one of them) and, without -l, one whose path names a unitig id the table does not have."""
    from oracle_lib import read_fasta
    names, seqs = read_fasta(info["sr"])
    piece = max(seqs, key=len)[:3000]
    path = os.path.join(tmp, "sr_edges%d.fa" % unknown_id)
    with open(path, "w") as f:
        f.write(open(info["sr"]).read())
        f.write(">contig_x\n%s\n" % piece)
        f.write(">contig_y rc\n%s\n" % piece[::-1].translate(str.maketrans("ACGT", "TGCA")))
        if unknown_id:
            f.write(">999999F_998877R\n%s\n" % seqs[1][:3000])
    return path


def run_fixture(name, parts):
    """Every alignment variant of one input, each result printed in every format on the device and on the host;
    with `parts`, the index is cut into 3-4 parts."""
    import pacbio_b200 as pb
    from oracle_lib import gen_synth
    tmp = os.environ["MR_COORDS_TMP"]
    if name == "big":
        info = gen_synth(os.path.join(tmp, "crd_big"), 1500000, coverage=4, read_len=8000, seed=77, repeat_frac=0.15)
        mer, psa, k = 15, 13, 41
    else:
        cfg = json.load(open(os.path.join(GOLD, name + ".json")))["config"]
        info = gen_synth(os.path.join(tmp, "crd_" + name), **cfg["gen"])
        mer, psa, k = cfg["mer"], cfg["psa_min"], cfg["unitig_k"]
    if parts:
        nbases = sum(len(l) - 1 for l in open(info["sr"]) if not l.startswith(">"))
        os.environ["MR_INDEX_PART_BASES"] = str(max(1024, nbases // 3 + 1000))
    H = host_lib()
    ulen = np.loadtxt(info["unitigs_len"], dtype=np.int64)[:, 1]
    reads = pb.Reads(info["reads"])
    rng = random.Random(3)
    names = reads.names + ["empty_read", "short_read", "random_read"]
    seqs = [reads.bases[int(reads.starts[i]):int(reads.starts[i + 1])].tobytes().decode() for i in range(reads.nreads)]
    seqs += ["", "ACGT", "".join(rng.choice("ACGT") for _ in range(3000))]
    reads = pb.Reads(names=names, seqs=seqs)
    read_len = np.diff(reads.starts.astype(np.int64))
    seen = dict(zero_rows=0, empty_read=0, bwd_path=0, bwd_nopath=0, no_info=0, rows=0)
    ctx1, ctx2 = pb.Context(0), pb.Context(0)
    for lk in (True, False):
        sr = pb.SuperReads(with_edge_super_reads(info, tmp, unknown_id=not lk))
        srn = ctx1.sr_names(sr.names, sr.unitig_ids, sr.unitig_off)
        idx = ctx1.index(sr, psa, mer, unitig_len=ulen if lk else None)
        assert idx.parts() in ((3, 4) if parts else (1,)), idx.parts()
        base = dict(unitigs_k=k if lk else 0, matching_bases=0.17, matching_mers=0.0, run_graph=0)
        runs = [(ctx, dict(base, forward=fwd), "fwd %d" % fwd) for fwd in (0, 1) for ctx in (ctx1, ctx2)]
        runs += [(ctx1, dict(base, max_match=1), "--max-match"), (ctx2, dict(base, window_size=2), "--window-size 2"),
                 (ctx1, dict(base, fine_mer=psa), "-F %d" % psa)]
        if lk:                                          # a result that also carries the overlap graph
            runs.append((ctx2, dict(base, run_graph=1, forward=1), "run_graph"))
        for ctx, kw, what in runs:
            res = ctx.align(idx, reads, pb.default_params(**kw), keep=True)
            compare(ctx, H, res, srn, sr.names, sr.unitig_ids, sr.unitig_off, reads.names, read_len,
                    "%s %s %s" % (name, "-l" if lk else "no -l", what))
            rc = res.read_coords.astype(np.int64)
            seen["zero_rows"] += int(np.sum(np.diff(rc) == 0))
            seen["empty_read"] += int(rc[-3] == rc[-4])
            seen["rows"] += res.ncoords
            seen["no_info"] += int(np.sum(res.info_len == 0))
            for row in range(res.ncoords):
                if res.use_bwd[row]:
                    seen["bwd_path" if len(sr.paths[res.sr[row]]) else "bwd_nopath"] += 1
            res.close()
        srn.close(); idx.close()
    ctx1.close(); ctx2.close()
    print("SEEN " + json.dumps(seen))


pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]


@pytest.mark.parametrize("parts", [False, True], ids=["one_part", "index_parts"])
@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3", "big"])
def test_device_coords_equal_the_host_formatter(tmpdir_session, name, parts):
    """synth_g1..3 and the 1.5 Mbp / 15 % repeat input, with and without -l -k, forward on and off, --max-match,
    --window-size 2 and -F, on two contexts sharing one index, each result in all four compact x -0 formats; with
    an index cut into parts when `parts`."""
    env = dict(os.environ, MR_COORDS_TMP=tmpdir_session)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "fixture", name, str(int(parts))], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1700)
    assert r.returncode == 0, (r.stdout.decode()[-3000:] + r.stderr.decode()[-3000:])
    seen = json.loads(r.stdout.decode().split("SEEN ")[-1])
    for case in ("zero_rows", "empty_read", "bwd_path", "bwd_nopath", "no_info"):
        assert seen[case] > 0, (case, seen)
    assert seen["rows"] > 200, seen


# ---- hand-made rows through mr_graph_batch ------------------------------------------------------------------------
RARE = [1e-5, 9.999995e-05, 9.9999949e-05, 0.0001, 999999.5, 999999.4, 1e6, 1234565.0, 1234575.0, 12345.25, 0.5, 2.5,
        0.0, -0.0, float("inf"), float("-inf"), float("nan"), -float("nan"), 1e300, -1e-300, 5e-324, 123456789.0,
        -1.5e-7, 1.7976931348623157e308]


def make_rows(seed, k=21):
    """Rows whose stretch / offset / avg_err are the doubles the aligner rarely makes, over a path table with empty
    paths (names that do not parse) and rows read backward."""
    rng = random.Random(seed)
    nu = 30
    ulen = [rng.choice([25, 60, 150, 400]) for _ in range(nu)]
    paths, sr_names = [[]], ["no_path_here"]
    for i in range(40):
        p = [rng.randrange(nu) * 2 + rng.randrange(2) for _ in range(rng.randrange(1, 6))]
        paths.append(p)
        sr_names.append("_".join("%d%s" % (x >> 1, "R" if x & 1 else "F") for x in p))
    paths.append([]); sr_names.append("another name with blanks")
    path_off = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.uint64)
    path_ids = np.array([x for p in paths for x in p], dtype=np.uint32)
    cols = {c: [] for c in ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "sr",
                            "rn", "use_bwd", "stretch", "offset", "avg_err", "info_off", "info_len")}
    kinfo, read_coords, read_len, names = [], [0], [], []
    for r, n in enumerate([0, 1, 3, 0, 7, 12, 30] + [rng.randrange(0, 10) for _ in range(30)]):
        for _ in range(n):
            p = rng.randrange(len(paths))
            rs = rng.randrange(1, 5000)
            cols["rs"].append(rs); cols["re"].append(rs + rng.randrange(0, 2000))
            cols["qs"].append(rng.randrange(1, 50)); cols["qe"].append(rng.randrange(100, 3000))
            cols["nb_mers"].append(rng.randrange(-5, 400))
            for c in ("pb_cons", "sr_cons", "pb_cover", "sr_cover"):
                cols[c].append(rng.randrange(2 ** 32) if rng.random() < 0.05 else rng.randrange(1000))
            cols["ql"].append(rng.randrange(100, 9000)); cols["sr"].append(p)
            cols["rn"].append(rng.randrange(2)); cols["use_bwd"].append(rng.randrange(2))
            for c in ("stretch", "offset", "avg_err"):
                cols[c].append(rng.choice(RARE) if rng.random() < 0.5 else rng.uniform(-3000, 3000))
            ilen = 2 * len(paths[p]) - 1 if paths[p] and rng.random() < 0.8 else 0
            cols["info_off"].append(len(kinfo)); cols["info_len"].append(ilen)
            kinfo += [rng.randrange(-3, 300) for _ in range(ilen)]
        read_coords.append(read_coords[-1] + n)
        read_len.append(rng.choice([0, rng.randrange(1, 20000)]))
        names.append("read%d/%d_%d" % (r, seed, n))
    rows = {c: np.array(v) for c, v in cols.items()}
    rows["read_coords"] = np.array(read_coords, dtype=np.uint64)
    rows["kmers_info"] = np.array(kinfo or [0], dtype=np.int32)
    rows["bases_info"] = np.array(kinfo or [0], dtype=np.int32) * 3 - 7
    return dict(rows=rows, read_len=np.array(read_len), names=names, path_ids=path_ids, path_off=path_off,
                sr_names=sr_names, ulen=np.array(ulen, dtype=np.int32), k=k)


def test_hand_made_rows_with_rare_doubles():
    import pacbio_b200 as pb
    H = host_lib()
    ctx = pb.Context(0)
    fields = set()
    for seed in range(4):
        d = make_rows(seed)
        srn = ctx.sr_names(d["sr_names"], d["path_ids"], d["path_off"])
        res = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], pb.default_params(unitigs_k=d["k"]))
        texts = compare(ctx, H, res, srn, d["sr_names"], d["path_ids"], d["path_off"], d["names"], d["read_len"],
                        "seed %d" % seed)
        for line in texts[(True, False)].split(b"\n"):
            if line and not line.startswith(b">"):
                fields.update(line.split()[11:14])
        res.close(); srn.close()
    ctx.close()
    for tok in (b"1e-05", b"9.99999e-05", b"0.0001", b"1e+06", b"999999", b"1.23456e+06", b"1.23458e+06", b"12345.2",
                b"0.5", b"2.5", b"0", b"-0", b"inf", b"-inf", b"1e+300", b"-1e-300", b"4.94066e-324"):
        assert tok in fields, (tok, sorted(fields)[:80])
    assert b"nan" in fields and b"-nan" in fields


# ---- the reference's own coords files -----------------------------------------------------------------------------
def parse_coords(path):
    """A compact coords file the way coords_file::next_batch (host_common.cpp) reads it: the rows' columns, one path
    table entry per row (its printed name), the reads' names and lengths (Rlen of the first row)."""
    import pacbio_b200 as pb
    lines = open(path, "rb").read().split(b"\n")
    i = 0
    while not lines[i].startswith(b">"):
        i += 1
    cols = {c: [] for c in ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "sr",
                            "rn", "use_bwd", "stretch", "offset", "avg_err", "info_off", "info_len")}
    kinfo, binfo, read_coords, read_len, names, sr_names, paths = [], [], [0], [], [], [], []
    while i < len(lines) and lines[i].startswith(b">"):
        head = lines[i][1:]
        n = int(head.split(b" ", 1)[0])
        names.append(head.split(b" ", 1)[1] if b" " in head else b"")
        for j in range(n):
            f = lines[i + 1 + j].split(b" ")
            for c, v in zip(("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover"), f[:9]):
                cols[c].append(int(v))
            if j == 0:
                read_len.append(int(f[9]))
            cols["ql"].append(int(f[10]))
            for c, v in zip(("stretch", "offset", "avg_err"), f[11:14]):
                cols[c].append(float(v))
            sr_names.append(f[14])
            paths.append(pb.api.parse_sr_name(f[14].decode()))
            cols["sr"].append(len(sr_names) - 1); cols["rn"].append(0); cols["use_bwd"].append(0)
            cols["info_off"].append(len(kinfo)); cols["info_len"].append(len(f) - 15)
            for pair in f[15:]:
                a, b = pair.split(b":")
                kinfo.append(int(a)); binfo.append(int(b))
        read_coords.append(read_coords[-1] + n)
        i += 1 + n
    rows = {c: np.array(v) for c, v in cols.items()}
    rows["read_coords"] = np.array(read_coords, dtype=np.uint64)
    rows["kmers_info"] = np.array(kinfo or [0], dtype=np.int32)
    rows["bases_info"] = np.array(binfo or [0], dtype=np.int32)
    path_off = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.uint64)
    path_ids = np.array([x for p in paths for x in p], dtype=np.uint32)
    header = b"".join(l + b"\n" for l in lines[:lines.index(next(l for l in lines if l.startswith(b">")))])
    return rows, read_len, names, sr_names, path_ids, path_off, header


@pytest.mark.parametrize("golden", ["synth_g1.coords.txt", "synth_g2.coords.txt", "synth_g3.coords.txt",
                                    "synth_g1.fine11.coords.txt", "synth_g3.fine12.coords.txt"])
def test_reference_coords_files_round_trip(golden):
    """The reference wrote these files; their rows go through mr_graph_batch and come back out of mr_coords_records
    byte for byte (%g with 6 digits reprints its own output after strtod)."""
    import pacbio_b200 as pb
    path = os.path.join(GOLD, golden)
    rows, read_len, names, sr_names, path_ids, path_off, header = parse_coords(path)
    ulen = np.full(int(path_ids.max()) + 1 if len(path_ids) else 1, 100, dtype=np.int32)
    ctx = pb.Context(0)
    srn = ctx.sr_names(sr_names, path_ids, path_off)
    res = ctx.graph(rows, read_len, path_ids, path_off, ulen, pb.default_params(unitigs_k=41))
    text = ctx.coords_records(res, names, sr_names=srn)
    res.close(); srn.close(); ctx.close()
    assert header + text == open(path, "rb").read()


# ---- refusals -----------------------------------------------------------------------------------------------------
def test_refusals():
    import pacbio_b200 as pb
    ctx = pb.Context(0)
    d = make_rows(11)
    srn = ctx.sr_names(d["sr_names"], d["path_ids"], d["path_off"])
    params = pb.default_params(unitigs_k=d["k"])
    first = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
    second = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
    with pytest.raises(pb.MrError, match="error -1: mr_coords_records: the result is not the latest result of this context"):
        ctx.coords_records(first, d["names"], sr_names=srn)
    assert ctx.coords_records(second, d["names"], sr_names=srn)
    other = pb.Context(0)
    with pytest.raises(pb.MrError, match="error -1: mr_coords_records: the result is not the latest"):
        other.coords_records(second, d["names"], sr_names=srn)
    # names that stop short of the rows' super-reads
    few = ctx.sr_names(d["sr_names"][:5], d["path_ids"][:int(d["path_off"][5])], d["path_off"][:6])
    with pytest.raises(pb.MrError, match=r"error -1: mr_coords_records: row \d+ refers to a super-read that the names do "
                                         r"not have \(5 super-reads\)"):
        ctx.coords_records(second, d["names"], sr_names=few)
    assert ctx.coords_records(second, d["names"], sr_names=srn)          # the context is still usable
    if gpu_count() > 1:
        far = pb.Context(1)
        far_names = far.sr_names(d["sr_names"], d["path_ids"], d["path_off"])
        with pytest.raises(pb.MrError, match="error -1: mr_coords_records: the super-read names live on another device"):
            ctx.coords_records(second, d["names"], sr_names=far_names)
        far_names.close(); far.close()
    for x in (first, second, few, srn):
        x.close()
    other.close(); ctx.close()


def gpu_count():
    r = subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
    return r.stdout.decode().count("GPU ") if r.returncode == 0 else 1


# ---- the tool -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env", [dict(MR_BATCH_BASES="150000", MR_STREAMS="2"), dict(MR_BATCH_BASES="150000", MR_GPUS="2")],
                         ids=["two_streams", "two_gpus"])
def test_jf_aligner_device_path_equals_the_host_path(tmpdir_session, tmp_path, env):
    """jf_aligner prints on the device unless --details is given; the coords files of the two paths are identical,
    over several batches, with and without --compact, -0 and -l -k."""
    from oracle_lib import gen_synth
    if "MR_GPUS" in env and gpu_count() < 2:
        pytest.skip("one GPU")
    info = gen_synth(os.path.join(tmpdir_session, "crd_tool"), 300000, coverage=4, read_len=4000, seed=31, repeat_frac=0.1)
    e = dict(os.environ, **env)
    for extra in ([], ["--compact"], ["-0"], ["--compact", "-0"], ["-l", info["unitigs_len"], "-k", "41", "-0"]):
        base = [JFA, "-s", "1M", "-m", "15", "-B", "17", "-r", info["sr"], "-p", info["reads"]] + extra
        dev, host = str(tmp_path / "dev.txt"), str(tmp_path / "host.txt")
        subprocess.run(base + ["--coords", dev], check=True, env=e)
        subprocess.run(base + ["--coords", host, "--details", str(tmp_path / "details.txt")], check=True, env=e)
        a, b = open(dev, "rb").read(), open(host, "rb").read()
        assert a == b and len(a) > 10000, extra


if __name__ == "__main__":
    if sys.argv[1] == "fixture":
        run_fixture(sys.argv[2], sys.argv[3] == "1")
