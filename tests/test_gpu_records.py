"""Mega-read records printed on the device (mr_records, Context.records) against the host formatter
(mrh::format_mega_reads, the printer the tools used before and still use for --dot) on the same result, byte for
byte, in one process."""
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
CMR = os.path.join(ROOT, "pacbio_b200", "bin", "create_mega_reads")
VARIANTS = [(tiling, trim) for tiling in (0, 1, 2, 3) for trim in (0, 1)]


def host_lib():
    H = C.CDLL(os.path.join(ROOT, "pacbio_b200", "libmegareads_host.so"))
    H.mrh_format_records.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_char_p,
                                     C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_uint64), C.c_char_p, C.c_size_t]
    H.mrh_free.argtypes = [C.c_void_p]
    return H


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def host_records(H, res, path_ids, path_off, ulen, names, read_len, rp, useq=None, uoff=None):
    """What mrh::format_mega_reads prints for the result; raises RuntimeError with its message."""
    ids = np.ascontiguousarray(path_ids if len(path_ids) else [0], dtype=np.uint32)
    off = np.ascontiguousarray(path_off, dtype=np.uint64)
    ul = np.ascontiguousarray(ulen, dtype=np.int32)
    enc = [n.encode() for n in names]
    noff = np.concatenate([[0], np.cumsum([len(n) for n in enc])]).astype(np.uint64)
    starts = np.concatenate([[0], np.cumsum(np.asarray(read_len, dtype=np.uint64))]).astype(np.uint64)
    uo = np.ascontiguousarray(uoff, dtype=np.uint64) if useq is not None else None
    out, size, err = C.c_void_p(), C.c_uint64(), C.create_string_buffer(300)
    rc = H.mrh_format_records(res.h, ptr(ids), ptr(off), len(off) - 1, ptr(ul), len(ul), useq,
                              ptr(uo) if uo is not None else None, b"".join(enc), ptr(noff), ptr(starts), C.byref(rp),
                              C.byref(out), C.byref(size), err, 300)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    text = C.string_at(out, size.value) if size.value else b""
    H.mrh_free(out)
    return text


def compare(ctx, H, res, path_ids, path_off, ulen, names, read_len, k, useq, uoff, unitigs, what, **rp_kw):
    """Every tiling x trim, with and without sequences: device bytes == host bytes.  Returns the texts."""
    import pacbio_b200 as pb
    texts = {}
    for tiling, trim in VARIANTS:
        rp = pb.records_params(k, tiling=tiling, trim=trim, **rp_kw)
        for u in (None, unitigs):
            want = host_records(H, res, path_ids, path_off, ulen, names, read_len, rp,
                                useq if u is not None else None, uoff)
            got = ctx.records(res, names, rp, u)
            if got != want:
                a, b = got.split(b"\n"), want.split(b"\n")
                i = next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), min(len(a), len(b)))
                raise AssertionError("%s tiling %d trim %d %s: line %d differs:\n device %r\n host   %r" % (
                    what, tiling, trim, "-u" if u is not None else "-l", i, a[i][:300] if i < len(a) else None,
                    b[i][:300] if i < len(b) else None))
            texts[(tiling, trim, u is not None)] = got
    return texts


def run_fixture(name):
    """The aligner's results of one input, on two contexts sharing one index and one mr_unitigs."""
    import pacbio_b200 as pb
    from oracle_lib import gen_synth
    tmp = os.environ["MR_RECORDS_TMP"]
    if name == "big":
        info = gen_synth(os.path.join(tmp, "rec_big"), 1500000, coverage=4, read_len=8000, seed=77, repeat_frac=0.15)
        mer, psa, k = 15, 13, 41
    else:
        cfg = json.load(open(os.path.join(GOLD, name + ".json")))["config"]
        info = gen_synth(os.path.join(tmp, "rec_" + name), **cfg["gen"])
        mer, psa, k = cfg["mer"], cfg["psa_min"], cfg["unitig_k"]
    H = host_lib()
    sr = pb.SuperReads(info["sr"])
    _, useq, uoff = pb.api.load_fasta(info["unitigs"])
    ulen = np.diff(uoff.astype(np.int64)).astype(np.int32)
    ctx1, ctx2 = pb.Context(0), pb.Context(0)
    idx = ctx1.index(sr, psa, mer, unitig_len=ulen)
    U = ctx1.unitigs(useq.tobytes(), uoff)
    reads = pb.Reads(info["reads"])
    read_len = np.diff(reads.starts.astype(np.int64))
    useq_b = useq.tobytes()
    lines = 0
    for bases in (0, 1):
        params = pb.default_params(unitigs_k=k, run_graph=1, bases=bases, forward=1, matching_bases=0.17, matching_mers=0.0)
        for ctx in (ctx1, ctx2):
            res = ctx.align(idx, reads, params, keep=True)
            texts = compare(ctx, H, res, sr.unitig_ids, sr.unitig_off, ulen, reads.names, read_len, k, useq_b, uoff, U,
                            "%s -b %d" % (name, bases))
            lines += texts[(0, 0, False)].count(b"\n")
            res.close()
    U.close(); idx.close(); ctx1.close(); ctx2.close()
    print("lines %d" % lines)


def routes_env(big):
    env = dict(os.environ)
    if big:
        env.update(MR_BIG_ROWS="3", MR_HUGE_ROWS="6")
    return env


pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]


@pytest.mark.parametrize("wide", [False, True], ids=["default_routes", "wide_routes"])
@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3", "big"])
def test_device_records_equal_the_host_formatter(tmpdir_session, name, wide):
    """synth_g1..3 and the 1.5 Mbp / 15 % repeat input, every tiling x trim x -b x (-l | -u), with the default
    thresholds and with MR_BIG_ROWS / MR_HUGE_ROWS lowered so that nearly every read takes the warp-per-read route."""
    env = routes_env(wide)
    env["MR_RECORDS_TMP"] = tmpdir_session
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "fixture", name], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=1700)
    assert r.returncode == 0, (r.stdout.decode()[-3000:] + r.stderr.decode()[-3000:])
    assert int(r.stdout.decode().split("lines")[-1]) > 50


# ---- hand-made rows through mr_graph_batch ------------------------------------------------------------------------
SPECIAL = [1e12, 1e300, float("inf"), float("-inf"), float("nan")]


def make_rows(seed, k=21):
    """Seeded rows for mr_graph_batch: unitig paths of 0-6 unitigs (some unitigs shorter than k - 1), reads of 0 to
    700 rows drawn from a few positions and scores (ties), stretch / offset values that make implied positions of
    1e12, 1e300, +-inf and nan, rows with rs == re, kmers_info with zeros at both ends (what --trim match cuts)."""
    rng = random.Random(seed)
    nu = 40
    ulen = [rng.choice([5, 10, 19, 25, 60, 150, 400]) for _ in range(nu)]
    alphabet = "ACGTacgtN"
    useq = "".join("".join(rng.choice(alphabet) for _ in range(l)) for l in ulen).encode()
    uoff = np.concatenate([[0], np.cumsum(ulen)]).astype(np.uint64)
    paths = [[], [rng.randrange(nu) * 2]]
    for _ in range(60):
        paths.append([rng.randrange(nu) * 2 + rng.randrange(2) for _ in range(rng.randrange(1, 7))])
    path_off = np.concatenate([[0], np.cumsum([len(p) for p in paths])]).astype(np.uint64)
    path_ids = np.array([x for p in paths for x in p], dtype=np.uint32)
    cols = {c: [] for c in ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "sr",
                            "rn", "use_bwd", "stretch", "offset", "avg_err", "info_off", "info_len")}
    kinfo, read_coords, read_len, names = [], [0], [], []
    sizes = [0, 1, 2, 5, 9, 14, 17, 20, 30, 40, 700, 600] + [rng.randrange(0, 25) for _ in range(40)]
    for r, n in enumerate(sizes):
        rlen = rng.randrange(2000, 9000)
        special = n <= 16 and rng.random() < 0.5
        dead = r % 7 == 3                                   # every span negative: no candidate
        for i in range(n):
            p = rng.randrange(len(paths))
            ql = sum(ulen[x >> 1] for x in paths[p]) - max(0, len(paths[p]) - 1) * (k - 1)
            ql = max(ql, 30)
            rs = rng.choice([1, 100, 500, 1000, 2000, 3000]) + (rng.randrange(3) if n < 100 else 0)
            re = rs if rng.random() < 0.1 else rs + rng.choice([0, 50, 150, 400, 1200])
            if dead:
                rs, re = 1000, 995
            stretch = rng.choice([1.0, 1.0, 0.9, 1.1, -1.0])
            offset = float(rs - rng.randrange(0, 50))
            if special and rng.random() < 0.4:
                offset = rng.choice(SPECIAL)
            if rng.random() < 0.2:
                offset = -float(rng.randrange(0, 200))          # implied start below 1: trims the front
            cols["rs"].append(rs); cols["re"].append(re)
            cols["qs"].append(rng.randrange(1, 50)); cols["qe"].append(ql - rng.randrange(0, 50))
            cols["nb_mers"].append(rng.choice([20, 40, 40, 80]))
            for c in ("pb_cons", "sr_cons", "pb_cover", "sr_cover"):
                cols[c].append(rng.randrange(100))
            cols["ql"].append(ql); cols["sr"].append(p)
            cols["rn"].append(rng.randrange(2)); cols["use_bwd"].append(rng.randrange(2))
            cols["stretch"].append(stretch); cols["offset"].append(offset); cols["avg_err"].append(rng.random() * 3)
            nun = len(paths[p])
            ilen = 2 * nun - 1 if nun else 0
            cols["info_off"].append(len(kinfo)); cols["info_len"].append(ilen)
            for t in range(ilen):
                edge = t < 2 or t >= ilen - 2
                kinfo.append(0 if (edge and rng.random() < 0.6) else rng.randrange(1, 30))
        read_coords.append(read_coords[-1] + n)
        read_len.append(rlen)
        names.append("read%d/%d_%d" % (r, seed, n))
    rows = {c: np.array(v) for c, v in cols.items()}
    rows["read_coords"] = np.array(read_coords, dtype=np.uint64)
    rows["kmers_info"] = np.array(kinfo or [0], dtype=np.int32)
    rows["bases_info"] = np.array(kinfo or [0], dtype=np.int32) * 2
    return dict(rows=rows, read_len=np.array(read_len), names=names, path_ids=path_ids, path_off=path_off,
                ulen=np.array(ulen, dtype=np.int32), useq=useq, uoff=uoff, k=k)


def per_read_lines(text):
    out, cur = {}, None
    for line in text.split(b"\n"):
        if line.startswith(b">"):
            cur = line[1:].decode()
            out[cur] = []
        elif line:
            out[cur].append(line)
    return out


def test_hand_made_rows_through_the_graph_batch():
    """The cases the printer must get right, each asserted to occur.  (A greedy or weighted tiling that places nothing
    cannot occur: tile_greedy always places the first candidate, its covered set and placed list being empty; the
    printer's fallback to the candidates in tiling-sort order is reached only with no candidate at all.)"""
    import pacbio_b200 as pb
    H = host_lib()
    ctx = pb.Context(0)
    seen = dict(many=0, over500=0, no_candidate=0, special=set(), zero_span=0, trimmed=0, tied_lpath=0, tied_end=0,
                tied_weight=0, path0=0, path1=0, short_unitig=0)
    for seed in range(6):
        d = make_rows(seed)
        U = ctx.unitigs(d["useq"], d["uoff"])
        for bases in (0, 1):
            params = pb.default_params(unitigs_k=d["k"], run_graph=1, bases=bases)
            res = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
            texts = compare(ctx, H, res, d["path_ids"], d["path_off"], d["ulen"], d["names"], d["read_len"], d["k"],
                            d["useq"], d["uoff"], U, "seed %d -b %d" % (seed, bases), density=0.0, min_length=0.0)
            cands = per_read_lines(texts[(0, 0, False)])
            seen["many"] += sum(1 for v in cands.values() if len(v) > 16)
            seen["over500"] += sum(1 for v in cands.values() if len(v) > 500)
            rows_per_read = np.diff(d["rows"]["read_coords"].astype(np.int64))
            seen["no_candidate"] += sum(1 for n, c in zip(d["names"], rows_per_read) if c > 0 and n not in cands)
            for v in cands.values():
                for line in v:
                    f = line.split()
                    for tok in f[:2]:
                        if tok in (b"inf", b"-inf", b"nan", b"-nan") or len(tok) > 15:
                            seen["special"].add(tok if len(tok) <= 15 else b"huge")
                    seen["zero_span"] += f[2] == f[3]
            seen["trimmed"] += texts[(0, 0, False)] != texts[(0, 1, False)]
            short = {i for i, l in enumerate(d["ulen"]) if l < d["k"] - 1}
            for v in cands.values():
                f = [line.split() for line in v]
                if len(v) > 16:                 # ties among more candidates than the insertion-sort range of std::sort
                    seen["tied_lpath"] += len({x[6] for x in f}) < len(f)
                    seen["tied_end"] += len({x[3] for x in f}) < len(f)
                    # same lpath and span: same density, so the same weight
                    seen["tied_weight"] += len({(x[2], x[3], x[6]) for x in f}) < len(f)
                for x in f:
                    if len(x) == 9:             # no path name: a path of 0 unitigs
                        seen["path0"] += 1
                        continue
                    ids = [int(e[:-1]) for e in x[8].split(b"_")]
                    seen["path1"] += len(ids) == 1
                    seen["short_unitig"] += any(i in short for i in ids)
            res.close()
        U.close()
    ctx.close()
    for case in ("many", "over500", "no_candidate", "zero_span", "trimmed", "tied_lpath", "tied_end", "tied_weight", "path0",
                 "path1", "short_unitig"):
        assert seen[case], (case, seen)
    assert {b"inf", b"-inf", b"huge"} <= seen["special"] and (b"nan" in seen["special"] or b"-nan" in seen["special"]), seen


def test_records_of_a_result_that_is_not_the_latest_are_refused():
    import pacbio_b200 as pb
    ctx = pb.Context(0)
    d = make_rows(11)
    params = pb.default_params(unitigs_k=d["k"], run_graph=1)
    first = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
    second = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
    rp = pb.records_params(d["k"], density=0.0, min_length=0.0)
    with pytest.raises(pb.MrError, match="error -1: mr_records: the result is not the latest"):
        ctx.records(first, d["names"], rp)
    assert ctx.records(second, d["names"], rp)
    other = pb.Context(0)
    with pytest.raises(pb.MrError, match="error -1"):
        other.records(second, d["names"], rp)
    for x in (first, second):
        x.close()
    other.close()
    ctx.close()


def test_unitig_id_missing_from_the_sequences_is_refused():
    """A unitig of a printed path that the -u sequences do not have: MR_EINVAL with the host formatter's message."""
    import pacbio_b200 as pb
    H = host_lib()
    ctx = pb.Context(0)
    d = make_rows(3)
    params = pb.default_params(unitigs_k=d["k"], run_graph=1)
    res = ctx.graph(d["rows"], d["read_len"], d["path_ids"], d["path_off"], d["ulen"], params)
    short = ctx.unitigs(d["useq"][:int(d["uoff"][5])], d["uoff"][:6])           # unitigs 0-4 only
    rp = pb.records_params(d["k"], density=0.0, min_length=0.0)
    with pytest.raises(pb.MrError, match="error -1: unitig id of a super-read name is not in the -u file"):
        ctx.records(res, d["names"], rp, short)
    with pytest.raises(RuntimeError, match="unitig id of a super-read name is not in the -u file"):
        host_records(H, res, d["path_ids"], d["path_off"], d["ulen"][:5], d["names"], d["read_len"], rp,
                     d["useq"][:int(d["uoff"][5])], d["uoff"][:6])
    res.close(); short.close(); ctx.close()


def test_tools_refuse_an_unknown_unitig_id_as_before(tmpdir_session, tmp_path):
    """A super-read name with a unitig id that the -u file does not have: the tools never reach the printer with it.
    mr_index_create / mr_align_batch and mr_graph_batch refuse such a table first, so create_mega_reads and
    longest_path_overlap_graph2 exit 1 with the message they printed before the records moved to the GPU."""
    from oracle_lib import gen_synth, read_fasta
    info = gen_synth(os.path.join(tmpdir_session, "rec_unknown"), 100000, coverage=2, read_len=4000, seed=5)
    names, seqs = read_fasta(info["reads"])
    sr = str(tmp_path / "sr.fa")
    with open(sr, "w") as f:
        f.write(open(info["sr"]).read())
        f.write(">999999F\n%s\n" % seqs[0][:3000])
    common = ["-s", "1M", "-m", "15", "-k", "41", "-r", sr, "-p", info["reads"]]
    r = subprocess.run([CMR] + common + ["-u", info["unitigs"], "-o", str(tmp_path / "out.txt")], stderr=subprocess.PIPE)
    assert r.returncode == 1
    assert b"create_mega_reads: mr_align_batch: mr_align_batch: a super-read name refers to a k-unitig that the unitig " \
        b"table (-l/-u) does not have\n" in r.stderr, r.stderr
    coords = str(tmp_path / "coords.txt")
    subprocess.run([os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")] + common + ["-H", "--coords", coords], check=True)
    assert b"999999F" in open(coords, "rb").read()
    r = subprocess.run([os.path.join(ROOT, "pacbio_b200", "bin", "longest_path_overlap_graph2"), "-k", "41", "-u", info["unitigs"],
                        "-o", str(tmp_path / "lp.txt"), coords], stderr=subprocess.PIPE)
    assert r.returncode == 1
    assert b"longest_path_overlap_graph2: mr_graph_batch: mr_graph_batch: a path refers to a k-unitig that the unitig " \
        b"table does not have\n" in r.stderr, r.stderr


def test_dot_keeps_the_records(tmpdir_session, tmp_path):
    """create_mega_reads with --dot (host formatter) writes the same records as without it (device printer)."""
    from oracle_lib import gen_synth
    info = gen_synth(os.path.join(tmpdir_session, "rec_dot"), 200000, coverage=3, read_len=4000, seed=11, repeat_frac=0.1)
    common = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-t", "1", "-r", info["sr"], "-p", info["reads"]]
    for extra in ([], ["-T", "maximal", "--trim", "match"]):
        a, b, dot = str(tmp_path / "a.txt"), str(tmp_path / "b.txt"), str(tmp_path / "a.dot")
        subprocess.run(common + extra + ["-o", a, "--dot", dot], check=True)
        subprocess.run(common + extra + ["-o", b], check=True)
        assert open(a, "rb").read() == open(b, "rb").read() and os.path.getsize(a) > 1000
        assert os.path.getsize(dot) > 1000


if __name__ == "__main__":
    if sys.argv[1] == "fixture":
        run_fixture(sys.argv[2])
