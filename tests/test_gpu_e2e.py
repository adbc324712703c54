"""End-to-end GPU parity: the drop-in binaries (pacbio_b200/bin/{create_mega_reads,jf_aligner}),
which reach the device only through the C ABI, against
  * the reference's own CLI goldens (tests/golden/aligner_output),
  * fixtures produced by the reference itself (tests/golden/synth_*), and
  * the oracle port (and the compiled reference when present) on larger seeded inputs."""
import hashlib
import json
import os
import subprocess

import pytest

from oracle_lib import REF_CMR, gen_synth, have_ref, records

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
CMR = os.path.join(ROOT, "pacbio_b200", "bin", "create_mega_reads")
JFA = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
LPG = os.path.join(ROOT, "pacbio_b200", "bin", "longest_path_overlap_graph2")


def sha(b):
    return hashlib.sha256(b).hexdigest()


def run(cmd, **kw):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, **kw)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    return r


def reads_with_coords_ties(coords_path):
    """Reads whose coords contain an exact (rs, re, ql) tie.  There the reference's own output is not
    defined: the tie is ordered by unordered_map pointer hash + unstable sort (create_mega_reads.cc:74,
    SURVEY.md 0.7) and can flip which of two equal-score mega-reads survives the tiling."""
    ties, cur, seen = set(), None, None
    for line in open(coords_path):
        if line.startswith(">"):
            cur, seen = line.split()[1], set()
        else:
            f = line.split()
            key = (f[0], f[1], f[10])
            if key in seen:
                ties.add(cur)
            seen.add(key)
    return ties


def assert_same_records(got, want, tie_reads=(), what=""):
    diff = [k for k in set(got) | set(want) if got.get(k) != want.get(k)]
    hard = [k for k in diff if k[1:] not in tie_reads]
    assert not hard, "%s: %d of %d records differ, e.g. %s" % (what, len(hard), len(want), hard[:3])
    assert len(diff) <= max(2, len(want) // 100), "%s: too many tie-related differences (%d)" % (what, len(diff))


@pytest.mark.parametrize("forward", [False, True])
def test_reference_cli_goldens(tmp_path, forward):
    d = os.path.join(GOLD, "aligner_output")
    out = str(tmp_path / "coords")
    det = str(tmp_path / "details")
    cmd = [JFA, "-s", "10k", "-m", "17", "-r", os.path.join(d, "test_super_reads.fa"), "-p",
           os.path.join(d, "test_pacbio.fa"), "--stretch-cap", "200", "--coords", out, "--details", det]
    if forward:
        cmd += ["-l", os.path.join(d, "test_unitigs_lengths"), "-k", "65", "-f"]
    run(cmd)
    got = sorted(tuple(l.split()) for l in open(out).read().splitlines()[1:] if not l.startswith(">"))
    want = []
    for line in open(os.path.join(d, "coords_forward_expected" if forward else "coords_normal_expected")).read().splitlines()[1:]:
        f = line.split()
        want.append(tuple(f[:14]) + tuple(f[15:]))     # golden is the old non-compact layout (Rname column)
    assert got == sorted(want)
    # --details: the reference's golden file, line for line (the reference sorts them too: tests/wdiffn -p sort)
    golden = os.path.join(d, "details_forward_expected" if forward else "details_normal_expected")
    assert sorted(open(det).read().splitlines()) == sorted(open(golden).read().splitlines())


@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3"])
def test_reference_generated_fixtures(tmpdir_session, tmp_path, name):
    meta = json.load(open(os.path.join(GOLD, name + ".json")))
    cfg = meta["config"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_" + name), **cfg["gen"])
    for key, h in meta["inputs"].items():
        assert sha(open(info[key], "rb").read()) == h
    common = ["-s", "1M", "-m", str(cfg["mer"]), "--psa-min", str(cfg["psa_min"]), "-k", str(cfg["unitig_k"]),
              "-r", info["sr"], "-p", info["reads"]]
    out = str(tmp_path / "cmr.txt")
    run([CMR] + common + ["-l", info["unitigs_len"], "-t", "4", "-B", "17", "--max-count", "5000", "-d", "0.029", "-o", out])
    assert records(out) == records(os.path.join(GOLD, name + ".cmr.txt"))
    out_u = str(tmp_path / "cmr_u.txt")
    run([CMR] + common + ["-u", info["unitigs"], "-t", "2", "-o", out_u])
    assert sha(open(out_u, "rb").read()) == meta["cmr_with_sequences_sha256_t1"]     # byte-identical file
    out_c = str(tmp_path / "coords.txt")
    run([JFA] + common + ["-l", info["unitigs_len"], "-H", "--coords", out_c])
    assert records(out_c) == records(os.path.join(GOLD, name + ".coords.txt"))


@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3"])
def test_index_of_several_parts_reproduces_the_reference_fixtures(tmpdir_session, tmp_path, name):
    """The route for super-read sets of 2^32 bases or more (several index parts), forced on the
    fixture inputs: same bytes as the reference's file."""
    meta = json.load(open(os.path.join(GOLD, name + ".json")))
    cfg = meta["config"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_" + name), **cfg["gen"])
    nbases = sum(len(l) - 1 for l in open(info["sr"]) if not l.startswith(">"))
    env = dict(os.environ, MR_INDEX_PART_BASES=str(max(1024, nbases // 3 + 1000)), MR_TRACE="1")
    common = ["-s", "1M", "-m", str(cfg["mer"]), "--psa-min", str(cfg["psa_min"]), "-k", str(cfg["unitig_k"]),
              "-r", info["sr"], "-p", info["reads"]]
    out_u = str(tmp_path / "cmr_u.txt")
    r = run([CMR] + common + ["-u", info["unitigs"], "-t", "2", "-o", out_u], env=env)
    assert b"index parts: 3" in r.stderr or b"index parts: 4" in r.stderr, r.stderr.decode()[-500:]
    assert sha(open(out_u, "rb").read()) == meta["cmr_with_sequences_sha256_t1"]
    out_c = str(tmp_path / "coords.txt")
    run([JFA] + common + ["-l", info["unitigs_len"], "-H", "--coords", out_c], env={k_: v_ for k_, v_ in env.items() if k_ != "MR_TRACE"})
    assert records(out_c) == records(os.path.join(GOLD, name + ".coords.txt"))


@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3"])
def test_many_row_kernels_reproduce_the_reference_fixtures(tmpdir_session, tmp_path, name):
    """Reads with many coords rows (repeats) get a CTA instead of a warp in the coords-order and
    overlap-graph kernels; MR_BIG_ROWS=3 sends nearly every read of the fixtures down that path."""
    meta = json.load(open(os.path.join(GOLD, name + ".json")))
    cfg = meta["config"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_" + name), **cfg["gen"])
    # more than 3 rows: the edge-list graph kernels and the CTA ordering; up to 6 rows their sequential state lives in
    # shared memory, above in global scratch; up to 8 rows the orderings are bitonic sorts, above rankings by counting
    env = dict(os.environ, MR_BIG_ROWS="3", MR_HUGE_ROWS="6", MR_SORT_ROWS="8")
    common = ["-s", "1M", "-m", str(cfg["mer"]), "--psa-min", str(cfg["psa_min"]), "-k", str(cfg["unitig_k"]),
              "-r", info["sr"], "-p", info["reads"]]
    out_u = str(tmp_path / "cmr_u.txt")
    run([CMR] + common + ["-u", info["unitigs"], "-t", "2", "-o", out_u], env=env)
    assert sha(open(out_u, "rb").read()) == meta["cmr_with_sequences_sha256_t1"]
    out_c = str(tmp_path / "coords.txt")
    run([JFA] + common + ["-l", info["unitigs_len"], "-H", "--coords", out_c], env=env)
    assert records(out_c) == records(os.path.join(GOLD, name + ".coords.txt"))
    # the graph stage from a coords file (longest_path_overlap_graph2) through the same kernels
    out_lp = str(tmp_path / "lp.txt")
    run([LPG, "-k", str(cfg["unitig_k"]), "-l", info["unitigs_len"], "-o", out_lp, os.path.join(GOLD, name + ".coords.txt")], env=env)
    assert open(out_lp).read() == open(os.path.join(GOLD, name + ".lp.txt")).read()


FINE = {"synth_g1": [(11, True), (14, False)], "synth_g2": [(13, False)], "synth_g3": [(12, True)]}   # as in make_golden.py


@pytest.mark.parametrize("parts", [False, True], ids=["one_part", "several_parts"])
@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3"])
def test_fine_pass_matches_reference_fixture(tmpdir_session, tmp_path, name, parts):
    """-F (fine_aligner.cc): windows from the coarse rows, shorter mers looked up in the same suffix array (fine mer
    below, at and above --psa-min), accept-all chaining -- against the reference's own records; also with the
    super-reads cut into several index parts (the layout of a text of 2^32 bases or more)."""
    cfg = json.load(open(os.path.join(GOLD, name + ".json")))["config"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_" + name), **cfg["gen"])
    env = dict(os.environ)
    if parts:
        nbases = sum(len(l) - 1 for l in open(info["sr"]) if not l.startswith(">"))
        env["MR_INDEX_PART_BASES"] = str(max(1024, nbases // 3 + 1000))
    common = ["-s", "1M", "-m", str(cfg["mer"]), "--psa-min", str(cfg["psa_min"]), "-k", str(cfg["unitig_k"]),
              "-l", info["unitigs_len"], "-r", info["sr"], "-p", info["reads"]]
    for fine, with_coords in FINE[name]:
        out = str(tmp_path / "cmr.txt")
        run([CMR] + common + ["-F", str(fine), "-t", "2", "-o", out], env=env)
        assert open(out).read() == open(os.path.join(GOLD, "%s.fine%d.cmr.txt" % (name, fine))).read()
        if with_coords:
            out = str(tmp_path / "coords.txt")
            run([JFA] + common + ["-F", str(fine), "-H", "--coords", out], env=env)
            assert records(out) == records(os.path.join(GOLD, "%s.fine%d.coords.txt" % (name, fine)))


def test_fine_pass_larger_input_against_oracle(tmpdir_session, tmp_path, port):
    info = gen_synth(os.path.join(tmpdir_session, "e2e_fine_big"), 400000, coverage=4, read_len=5000, seed=37, repeat_frac=0.1)
    for fine, extra in ((12, []), (10, ["--max-match"])):
        out, want = str(tmp_path / "gpu.txt"), str(tmp_path / "port.txt")
        run([CMR, "-s", "1M", "-m", "15", "-k", "41", "-l", info["unitigs_len"], "-r", info["sr"], "-p", info["reads"],
             "-F", str(fine), "-o", out] + extra, env=dict(os.environ, MR_BATCH_BASES="300000"))
        port.run(0, info["sr"], info["reads"], info["unitigs_len"], want, 15, 41, unitigs_is_fasta=False, threads=8,
                 fine_mer=fine, max_match=bool(extra))
        got, exp = records(out), records(want)
        diff = [k for k in set(got) | set(exp) if got.get(k) != exp.get(k)]
        assert len(exp) > 200 and len(diff) <= max(2, len(exp) // 100), (len(diff), len(exp), diff[:3])


LP_VARIANTS = {"lp": [], "lp_maximal": ["-T", "maximal", "--trim", "match", "-b", "-O", "1.5", "-d", "0.01"]}   # as in make_golden.py


@pytest.mark.parametrize("variant", sorted(LP_VARIANTS))
@pytest.mark.parametrize("name", ["synth_g1", "synth_g2", "synth_g3"])
def test_longest_path_matches_reference_fixture(tmpdir_session, tmp_path, name, variant):
    """longest_path_overlap_graph2 (coords file -> overlap graph on the GPU -> mega-reads) against the
    reference binary's output on the same committed coords file, byte for byte."""
    cfg = json.load(open(os.path.join(GOLD, name + ".json")))["config"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_" + name), **cfg["gen"])
    out = str(tmp_path / "lp.txt")
    run([LPG, "-k", str(cfg["unitig_k"]), "-l", info["unitigs_len"], "-t", "3"] + LP_VARIANTS[variant] +
        ["-o", out, os.path.join(GOLD, name + ".coords.txt")])
    assert open(out).read() == open(os.path.join(GOLD, "%s.%s.txt" % (name, variant))).read()
    # small batches (several mr_graph_batch calls) give the same file
    out2 = str(tmp_path / "lp2.txt")
    run([LPG, "-k", str(cfg["unitig_k"]), "-l", info["unitigs_len"]] + LP_VARIANTS[variant] +
        ["-o", out2, os.path.join(GOLD, name + ".coords.txt")], env=dict(os.environ, MR_BATCH_ROWS="37"))
    assert open(out2).read() == open(out).read()


def test_longest_path_agrees_with_create_mega_reads(tmpdir_session, tmp_path):
    """jf_aligner --coords | longest_path_overlap_graph2 is the same pipeline as create_mega_reads cut in two at a text
    file; apart from the decimals lost in that file the two give the same mega-reads (same reads, same super-read paths)."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_lp_pipe"), 200000, coverage=4, read_len=4000, seed=29)
    common = ["-s", "1M", "-m", "15", "-k", "41", "-r", info["sr"], "-p", info["reads"]]
    coords, lp, cmr = (str(tmp_path / n) for n in ("coords.txt", "lp.txt", "cmr.txt"))
    run([JFA] + common + ["-l", info["unitigs_len"], "--coords", coords])
    run([LPG, "-k", "41", "-l", info["unitigs_len"], "-o", lp, coords])
    run([CMR] + common + ["-l", info["unitigs_len"], "-o", cmr])

    def paths(path):
        out, cur = {}, None
        for line in open(path):
            if line.startswith(">"):
                cur = out.setdefault(line.strip(), [])
            else:
                cur.append(line.split()[8])
        return out
    a, b = paths(lp), paths(cmr)
    assert len(b) > 100
    same = sum(1 for k in b if a.get(k) == b[k])
    assert same >= 0.98 * len(b), (same, len(b))


@pytest.mark.parametrize("tiling,trim,bases", [("greedy", "none", False), ("maximal", "match", False),
                                               ("weighted", "none", True), ("none", "match", False)])
def test_larger_input_against_oracle(tmpdir_session, tmp_path, port, tiling, trim, bases):
    info = gen_synth(os.path.join(tmpdir_session, "e2e_big"), 1500000, coverage=4, read_len=8000, seed=77,
                     repeat_frac=0.15, threads=4)
    out = str(tmp_path / "gpu.txt")
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-t", "4", "-T", tiling, "--trim", trim,
           "-r", info["sr"], "-p", info["reads"], "-o", out]
    if bases:
        cmd.append("-b")
    env = dict(os.environ, MR_BATCH_BASES="2000000")          # several batches
    if tiling == "maximal":
        env["MR_BIG_ROWS"] = "8"                              # reads with more than 8 rows through the many-row kernels
        env["MR_HUGE_ROWS"] = "20"
    run(cmd, env=env)
    want = str(tmp_path / "oracle.txt")
    if have_ref():
        run([REF_CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-t", "8", "-T", tiling, "--trim", trim,
             "-r", info["sr"], "-p", info["reads"], "-o", want] + (["-b"] if bases else []))
    else:
        port.run(0, info["sr"], info["reads"], info["unitigs"], want, 15, 41, threads=8, bases=bases,
                 tiling=["none", "greedy", "maximal", "weighted"].index(tiling), trim=1 if trim == "match" else 0)
    a, b = records(out), records(want)
    assert len(b) > 500
    diff = [k for k in set(a) | set(b) if a.get(k) != b.get(k)]
    assert not diff, "%d of %d records differ, e.g. %s" % (len(diff), len(b), diff[:3])


def test_max_match_text_against_reference(tmpdir_session, tmp_path, port):
    info = gen_synth(os.path.join(tmpdir_session, "e2e_mm"), 300000, coverage=4, read_len=5000, seed=9, repeat_frac=0.25)
    common = ["-s", "1M", "-m", "15", "-k", "41", "-l", info["unitigs_len"], "--max-match", "-r", info["sr"], "-p", info["reads"]]
    out, outc = str(tmp_path / "gpu.txt"), str(tmp_path / "gpu.coords")
    run([CMR] + common + ["-o", out])
    run([JFA] + common + ["-H", "--coords", outc])
    want, wantc = str(tmp_path / "want.txt"), str(tmp_path / "want.coords")
    if have_ref():
        from oracle_lib import REF_JFA
        run([REF_CMR] + common + ["-t", "4", "-o", want])
        run([REF_JFA] + common + ["-t", "1", "-H", "--coords", wantc])
    else:
        port.run(0, info["sr"], info["reads"], info["unitigs_len"], want, 15, 41, unitigs_is_fasta=False, max_match=True)
        port.run(1, info["sr"], info["reads"], info["unitigs_len"], wantc, 15, 41, unitigs_is_fasta=False, max_match=True)
    assert_same_records(records(outc), records(wantc), what="coords")
    assert_same_records(records(out), records(want), reads_with_coords_ties(outc), what="mega reads")


def test_oversized_batches_are_split(tmpdir_session, tmp_path):
    """A batch that exceeds a device limit is cut in halves by the host pipeline; the records do not change."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_split"), 200000, coverage=4, read_len=4000, seed=21)
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-l", info["unitigs_len"], "-r", info["sr"], "-p", info["reads"]]
    a, b = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
    run(cmd + ["-o", a])
    run(cmd + ["-o", b], env=dict(os.environ, MR_MAX_HITS="20000"))
    assert open(a).read() == open(b).read() and len(open(a).read()) > 1000


def test_several_batches_in_flight_keep_the_record_order(tmpdir_session, tmp_path):
    """MR_STREAMS contexts per GPU share one index; the formatter puts the batches back in input order."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_streams"), 200000, coverage=6, read_len=4000, seed=23)
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-l", info["unitigs_len"], "-r", info["sr"], "-p", info["reads"]]
    a, b = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
    run(cmd + ["-o", a], env=dict(os.environ, MR_STREAMS="1"))
    run(cmd + ["-o", b], env=dict(os.environ, MR_STREAMS="3", MR_BATCH_BASES="60000"))
    assert open(a).read() == open(b).read() and len(open(a).read()) > 1000


def test_index_cache_is_used_and_checked(tmpdir_session, tmp_path):
    """MR_INDEX_CACHE: the first run builds and saves, the second loads; a cache made from other super-reads is rebuilt."""
    a = gen_synth(os.path.join(tmpdir_session, "e2e_cache_a"), 150000, coverage=3, read_len=3000, seed=41)
    b = gen_synth(os.path.join(tmpdir_session, "e2e_cache_b"), 150000, coverage=3, read_len=3000, seed=42)
    cache = str(tmp_path / "index.cache")
    env = dict(os.environ, MR_INDEX_CACHE=cache)

    def go(info, out, env_):
        cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-r", info["sr"], "-p", info["reads"], "-o", out]
        return subprocess.run(cmd, env=env_, stderr=subprocess.PIPE, check=True).stderr.decode()

    plain, first, second, other = (str(tmp_path / n) for n in ("plain.txt", "first.txt", "second.txt", "other.txt"))
    go(a, plain, os.environ)
    assert "built and saved" in go(a, first, env) and os.path.getsize(cache) > 100000
    assert "loaded from" in go(a, second, env)
    assert open(plain).read() == open(first).read() == open(second).read() and len(open(plain).read()) > 1000
    assert "built and saved" in go(b, other, env)            # checksum mismatch: not used, replaced
    assert "loaded from" in go(b, other, env)


@pytest.mark.skipif(not have_ref(), reason="needs the compiled reference (oracle/_ref)")
def test_dot_file_matches_the_reference(tmpdir_session, tmp_path):
    """--dot: the overlap graph of every read as the reference writes it with -t 1 (overlap_graph.hpp:189-196,
    overlap_graph.cc:49-50,133-146,271): nodes, every overlap edge with the k-mers it shares, the printed paths in red."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_dot"), 200000, coverage=3, read_len=4000, seed=11, repeat_frac=0.1)
    common = ["-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-t", "1", "-r", info["sr"], "-p", info["reads"]]
    run([CMR] + common + ["-o", str(tmp_path / "gpu.txt"), "--dot", str(tmp_path / "gpu.dot")])
    run([REF_CMR] + common + ["-o", str(tmp_path / "ref.txt"), "--dot", str(tmp_path / "ref.dot")])
    assert records(str(tmp_path / "gpu.txt")) == records(str(tmp_path / "ref.txt"))

    def graphs(path):
        out, cur = {}, None
        for line in open(path):
            if line.startswith("digraph"):
                cur = line.split('"')[1]
                out[cur] = []
            elif cur is not None and line.strip() != "}":
                out[cur].append(line)
        return out
    g, w = graphs(str(tmp_path / "gpu.dot")), graphs(str(tmp_path / "ref.dot"))
    assert list(g) == list(w) and len(g) > 100
    same = sum(1 for k in g if g[k] == w[k])
    # a read whose coords hold an exact (rs, re, ql) tie numbers those nodes in the other order (SURVEY.md 0.7)
    assert same >= len(g) - max(2, len(g) // 50), "%d of %d graphs differ" % (len(g) - same, len(g))
    assert open(str(tmp_path / "gpu.dot")).read().count("}\n") == open(str(tmp_path / "ref.dot")).read().count("}\n")
    assert sum(1 for k in g for l in g[k] if "->" in l and "label=" in l) > 50


def test_tiles_staged_without_bulk_copies_give_the_same_records(tmpdir_session, tmp_path):
    """MR_NO_TMA=1: the read tiles reach shared memory through ordinary loads instead of the TMA engine's bulk copies."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_tma"), 300000, coverage=4, read_len=4000, seed=19, repeat_frac=0.1)
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-r", info["sr"], "-p", info["reads"]]
    a, b = str(tmp_path / "tma.txt"), str(tmp_path / "plain.txt")
    run(cmd + ["-o", a])
    run(cmd + ["-o", b], env=dict(os.environ, MR_NO_TMA="1"))
    assert open(a).read() == open(b).read() and len(open(a).read()) > 10000


@pytest.mark.parametrize("env", [{"MR_READ_SORT": "0"}, {"MR_GSORT_CAP": "32"}, {"MR_GSORT_CAP": "256"},
                                 {"MR_GSORT_THREADS": "1024"}, {"MR_GSORT_THREADS": "1024", "MR_GSORT_CAP": "1024"}])
def test_grouping_routes_give_the_same_records(tmpdir_session, tmp_path, env):
    """Hits are grouped by (read, super-read) one CTA per read: in shared memory when the read's hits fit (default for
    these inputs), cut into buckets by the top bits of the super-read index first when they do not, by passes out of
    global memory for a bucket that still does not fit (MR_GSORT_CAP lowers what fits: 32 sends whole buckets there);
    or by the device-wide radix sort (MR_READ_SORT=0).  The records are the same bytes, and the reference's on the fixture."""
    meta = json.load(open(os.path.join(GOLD, "synth_g1.json")))
    cfg = meta["config"]
    fix = gen_synth(os.path.join(tmpdir_session, "e2e_synth_g1"), **cfg["gen"])
    out_u = str(tmp_path / "cmr_u.txt")
    run([CMR, "-s", "1M", "-m", str(cfg["mer"]), "--psa-min", str(cfg["psa_min"]), "-k", str(cfg["unitig_k"]),
         "-r", fix["sr"], "-p", fix["reads"], "-u", fix["unitigs"], "-t", "2", "-o", out_u], env=dict(os.environ, **env))
    assert sha(open(out_u, "rb").read()) == meta["cmr_with_sequences_sha256_t1"]
    info = gen_synth(os.path.join(tmpdir_session, "e2e_group"), 300000, coverage=4, read_len=4000, seed=29, repeat_frac=0.15)
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-r", info["sr"], "-p", info["reads"]]
    a, b = str(tmp_path / "default.txt"), str(tmp_path / "route.txt")
    run(cmd + ["-o", a])
    run(cmd + ["-o", b], env=dict(os.environ, **env))
    assert open(a).read() == open(b).read() and len(open(a).read()) > 10000


def test_fastq_and_multiple_files(tmpdir_session, tmp_path, port):
    info = gen_synth(os.path.join(tmpdir_session, "e2e_fq"), 100000, coverage=3, read_len=3000, seed=5)
    from oracle_lib import read_fasta
    names, seqs = read_fasta(info["reads"])
    half = len(names) // 2
    fa, fq = str(tmp_path / "a.fa"), str(tmp_path / "b.fq")
    with open(fa, "w") as f:
        for n, s in zip(names[:half], seqs[:half]):
            f.write(">%s some comment\n" % n)
            for i in range(0, len(s), 61):
                f.write(s[i:i + 61] + "\n")
    with open(fq, "w") as f:
        for n, s in zip(names[half:], seqs[half:]):
            f.write("@%s\n%s\n+\n%s\n" % (n, s, "I" * len(s)))
    out = str(tmp_path / "gpu.txt")
    run([CMR, "-s", "1M", "-m", "15", "-k", "41", "-l", info["unitigs_len"], "-r", info["sr"], "-p", fa, "-p", fq, "-o", out])
    want = str(tmp_path / "port.txt")
    port.run(0, info["sr"], info["reads"], info["unitigs_len"], want, 15, 41, unitigs_is_fasta=False)
    assert records(out) == records(want)


@pytest.mark.skipif(bool(os.environ.get("MR_SKIP_BIG_TESTS")), reason="MR_SKIP_BIG_TESTS set (135 Mbp genome, ~1 minute of reference CPU time)")
def test_arabidopsis_size_index_against_reference(tmpdir_session, tmp_path, port):
    """BASELINE.json configs[2] index scale (135 Mbp genome, 270 M super-read bases, repeat-rich) on a
    subsample of reads.  The text of the GPU tool must equal the oracle port's (same canonical tie
    rule) and the reference's, except for reads whose coords hold an exact (rs, re, ql) tie."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_c3"), 135000000, coverage=0.06, read_len=10000, seed=44,
                     error=0.15, repeat_frac=0.1, threads=16)
    common = ["-s", "1M", "-m", "15", "-k", "41", "-r", info["sr"], "-p", info["reads"]]
    out = str(tmp_path / "gpu.txt")
    run([CMR] + common + ["-u", info["unitigs"], "-t", "8", "-o", out])
    coords = str(tmp_path / "gpu.coords")
    run([JFA] + common + ["-l", info["unitigs_len"], "-H", "--coords", coords])
    got = records(out)
    assert len(got) > 300
    want_port = str(tmp_path / "port.txt")
    port.run(0, info["sr"], info["reads"], info["unitigs"], want_port, 15, 41, threads=16)
    assert_same_records(got, records(want_port), what="vs oracle port")
    if have_ref():
        want = str(tmp_path / "ref.txt")
        run([REF_CMR] + common + ["-u", info["unitigs"], "-t", "16", "-o", want])
        assert_same_records(got, records(want), reads_with_coords_ties(coords), what="vs reference")


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs on the box (gpurun --gpus 2)")
def test_reads_sharded_over_two_gpus_give_the_same_records(tmpdir_session, tmp_path):
    """MR_GPUS=2: index replicated, batches dealt to the two devices, host gather; same records."""
    info = gen_synth(os.path.join(tmpdir_session, "e2e_2gpu"), 400000, coverage=6, read_len=5000, seed=23)
    cmd = [CMR, "-s", "1M", "-m", "15", "-k", "41", "-u", info["unitigs"], "-t", "4", "-r", info["sr"], "-p", info["reads"]]
    one, two = str(tmp_path / "one.txt"), str(tmp_path / "two.txt")
    env = dict(os.environ, MR_BATCH_BASES="300000")           # many small batches so that both devices get work
    run(cmd + ["-o", one], env=env)
    run(cmd + ["-o", two], env=dict(env, MR_GPUS="2"))
    a, b = records(one), records(two)
    assert len(a) > 300 and a == b
