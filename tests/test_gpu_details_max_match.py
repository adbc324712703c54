"""--max-match with parity taps on, and jf_aligner --max-match --details.  The taps hold the state the discard loop
(coarse_aligner.cc:42-60) leaves every (read, super-read) group in: both hit lists without the hits of the chains it
removed, and each list's latest chain.  They are checked against the oracle port (and the compiled reference when it
travelled to the box) read by read, and through the tool against the restatement of print_details in
tests/details_lib.py."""
import os
import subprocess
from collections import Counter

import numpy as np
import pytest

from details_lib import port_details
from oracle_lib import Ref, device_rows, gen_synth, have_ref, oracle_rows, read_fasta, records
from test_gpu_stages import CASES

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JFA = os.path.join(ROOT, "pacbio_b200", "bin", "jf_aligner")
GOLD = os.path.join(ROOT, "tests", "golden", "aligner_output")

COMP = str.maketrans("ACGTacgt", "TGCAtgca")


def revcomp(s):
    return s.translate(COMP)[::-1]


def max_match_reads(info):
    """The case's first reads plus reads built to drive the discard loop into each of its states."""
    _, seqs = read_fasta(info["reads"])
    _, srs = read_fasta(info["sr"])
    seqs = seqs[:40]
    s0 = seqs[0]
    seqs.append(s0[:700] + "NNNN" + s0[704:1500] + "n" + s0[1501:2400])   # N runs
    seqs += ["ACGT", ""]
    longs = [x for x in srs if len(x) > 2500][:8]
    for s in longs[:4]:
        seg = s[100:1300]
        seqs.append(seg + "ACGTTGCA" + seg + s[1300:2000])                   # the same segment twice: a secondary row
        seqs.append(seg + "A" + seg + "C" + seg)                              # three times: three rows
        seqs.append(seg + "ACGTTGCA" + s[2000:2060])        # a short piece left over: its chain fails the default filters
    # a segment and its reverse complement: forward and backward chains of the same length.  The row is built from the
    # forward chain, the backward one is dropped (pb_aligner.hpp:87-92), so the forward row is emitted a second time.
    # The pads shift the k-mer sampling of the first bases of a run (jf_aligner.hpp:113-123), which decides whether the
    # two chains come out exactly equal.
    for s in longs:
        seg = s[200:1400]
        seqs += [seg + pad + revcomp(seg) for pad in ("N", "NN", "NNN", "ACGTN")]
    longest = max(srs, key=len)
    seqs.append(longest[:6000])                                               # one chain of thousands of hits
    return seqs


def read_taps(res, r):
    """Read r's taps in the layout of the checkers' align_read: groups (sr, n_fwd, n_bwd, lis_fwd, lis_bwd), offsets, lis."""
    sel = res.tap_groups[:, 0] == r
    rows = res.tap_groups[sel]
    first = int(np.flatnonzero(sel)[0]) if len(rows) else 0
    off0, lis0 = int(res.tap_groups[:first, 2:4].sum()), int(res.tap_groups[:first, 4:6].sum())
    noff, nlis = int(rows[:, 2:4].sum()), int(rows[:, 4:6].sum())
    return rows[:, 1:], res.tap_offsets[off0:off0 + noff], res.tap_lis[lis0:lis0 + nlis]


def coverage(groups, rows, groups_before):
    """What the discard loop went through, from one read's final groups, its rows and its groups before any discard."""
    per_sr = Counter(row[0][12] for row in rows)
    before = {int(g[0]): g for g in groups_before}
    seen = set()
    if max(per_sr.values(), default=0) >= 3:
        seen.add("three or more rows")
    if len(set(rows)) < len(rows):
        seen.add("forward row emitted twice")
    for g in groups:
        sr, nf, nb, lf, lb = (int(x) for x in g)
        if not per_sr[sr]:
            continue
        if lf + lb > 0:
            seen.add("non-empty final chain")
        b = before[sr]
        if (nf == 0 < b[1]) or (nb == 0 < b[2]):
            seen.add("list emptied")
    if any(int(g[1] + g[2]) >= 2000 for g in groups_before):
        seen.add("thousands of hits")
    return seen


WANT = {"three or more rows", "forward row emitted twice", "non-empty final chain", "list emptied", "thousands of hits"}


@pytest.fixture(scope="module")
def ctx():
    import pacbio_b200 as pb
    c = pb.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module", params=CASES, ids=lambda c: c["name"])
def case(request, tmpdir_session, ctx, port):
    import pacbio_b200 as pb
    c = dict(request.param)
    gen = {k: c[k] for k in ("genome", "coverage", "read_len", "seed", "repeat_frac", "error", "mean_unitig") if k in c}
    info = gen_synth(os.path.join(tmpdir_session, "gpu_" + c["name"]), unitig_k=c["uk"], **gen)
    sr = pb.SuperReads(info["sr"])
    ul = np.loadtxt(info["unitigs_len"], dtype=np.int64)[:, 1]
    idx = ctx.index(sr, c["m"], c["k"], unitig_len=ul)
    hp = port.index_create(info["sr"], c["m"], c["k"])
    port.set_unitigs_lengths(hp, ul)
    seqs = max_match_reads(info)
    reads = pb.Reads(names=["r%d" % i for i in range(len(seqs))], seqs=seqs)
    yield dict(cfg=c, info=info, sr=sr, ul=ul, idx=idx, hp=hp, seqs=seqs, reads=reads)
    idx.close()
    port.index_destroy(hp)


def _align(ctx, idx, reads, p, taps):
    ctx.keep_taps(taps)
    try:
        return ctx.align(idx, reads, p)
    finally:
        ctx.keep_taps(False)


@pytest.mark.parametrize("filters", ["default", "accept_all"])
@pytest.mark.parametrize("forward,window", [(True, 1), (False, 1), (True, 3), (False, 3)])
def test_max_match_taps_match_oracle(case, ctx, port, forward, window, filters):
    """Every read's groups, hit lists and chains after the discard loop equal the port's (and the reference's); the rows
    with taps on equal the rows with taps off and the oracle's, doubles bit for bit."""
    import pacbio_b200 as pb
    c, seqs = case["cfg"], case["seqs"]
    uk = c["uk"] if forward else 0
    mb = 0.0 if filters == "accept_all" else 0.17
    p = pb.default_params(unitigs_k=uk, run_graph=0, forward=int(forward), window_size=window, max_match=1)
    p.matching_bases, p.matching_mers = mb, 0.0
    res = _align(ctx, case["idx"], case["reads"], p, True)
    prod = _align(ctx, case["idx"], case["reads"], p, False)
    kw = dict(unitigs_k=uk, forward=forward, window_size=window, matching_bases=mb, matching_mers=0.0)
    ap = port.aligner_create(case["hp"], max_match=True, **kw)
    ap0 = port.aligner_create(case["hp"], max_match=False, **kw)
    ref = ar = None
    if have_ref():
        ref = Ref()
        hr = ref.index_create(case["info"]["sr"], c["m"], c["k"])
        ref.set_unitigs_lengths(hr, case["ul"])
        ar = ref.aligner_create(hr, max_match=True, **kw)
    seen, total_rows = set(), 0
    for r, s in enumerate(seqs):
        o = port.align_read(ap, s)
        groups, offsets, lis = read_taps(res, r)
        assert np.array_equal(groups, o["groups"]), "groups of read %d" % r
        assert np.array_equal(offsets, o["offsets"]), "hit lists of read %d" % r
        assert np.array_equal(lis, o["lis"]), "chains of read %d" % r
        if ref:
            w = ref.align_read(ar, s)
            for key in ("groups", "offsets", "lis"):
                assert np.array_equal(w[key], o[key]), "reference %s of read %d" % (key, r)
        want = oracle_rows(o)
        got = device_rows(res, r, len(s))
        assert got == want, "coords of read %d" % r
        assert device_rows(prod, r, len(s)) == got, "coords of read %d without taps" % r
        total_rows += len(want)
        seen |= coverage(groups, got, port.align_read(ap0, s)["groups"])
    assert total_rows > 40
    # accept-all filters pass every row, so the loop only ends once both lists are empty
    want = WANT if filters == "default" else WANT - {"non-empty final chain"}
    assert seen == want, "not exercised: %s, unexpected: %s" % (sorted(want - seen), sorted(seen - want))
    port.aligner_destroy(ap)
    port.aligner_destroy(ap0)
    if ref:
        ref.aligner_destroy(ar)
        ref.index_destroy(hr)


def test_index_of_several_parts_gives_the_same_taps(case, ctx):
    """An index cut into several parts (MR_INDEX_PART_BASES, the layout of a text of 2^32 bases or more) leaves the
    lists and chains after the discard loop, and the rows, as they are with one part."""
    import pacbio_b200 as pb
    c = case["cfg"]
    os.environ["MR_INDEX_PART_BASES"] = str(max(1024, int(case["sr"].n / 3.3)))
    try:
        idx = ctx.index(case["sr"], c["m"], c["k"], unitig_len=case["ul"])
    finally:
        del os.environ["MR_INDEX_PART_BASES"]
    try:
        assert idx.parts() in (3, 4)
        p = pb.default_params(unitigs_k=c["uk"], run_graph=0, max_match=1)
        want, got = [_align(ctx, ix, case["reads"], p, True) for ix in (case["idx"], idx)]
        assert len(want.tap_groups) > 100 and want.ncoords > 40
        for f in ("tap_groups", "tap_offsets", "tap_lis"):
            assert np.array_equal(getattr(got, f), getattr(want, f)), f
        for r, s in enumerate(case["seqs"]):
            assert device_rows(got, r, len(s)) == device_rows(want, r, len(s)), "coords of read %d" % r
    finally:
        idx.close()


def _run(cmd, env=None):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600, env=env)
    assert r.returncode == 0, r.stderr.decode()[-2000:]


def _sorted_lines(path):
    return sorted(open(path).read().splitlines())


def _details_run(tmp_path, port, cmd, env, sr, reads, unitigs_len, mer, unitig_k, forward, **kw):
    """jf_aligner with --details and without: the coords files are the same bytes, the coords are the port's, and the
    details file holds the lines the reference's print_details writes for the port's final groups."""
    coords, coords_plain, details = (str(tmp_path / n) for n in ("coords", "coords_plain", "details"))
    _run(cmd + ["--coords", coords, "--details", details], env)
    _run(cmd + ["--coords", coords_plain], env)
    assert open(coords, "rb").read() == open(coords_plain, "rb").read()
    want_coords = str(tmp_path / "port_coords")
    port.run(1, sr, reads, unitigs_len, want_coords, mer, unitig_k, unitigs_is_fasta=False, forward=forward,
             max_match=True, threads=4, **kw)
    assert records(coords) == records(want_coords)
    want, single = _port_details(port, sr, reads, mer, forward, True, **kw), _port_details(port, sr, reads, mer, forward, False, **kw)
    got = _sorted_lines(details)
    assert got == sorted(want), "%d of %d details lines differ" % (len(set(got) ^ set(want)), len(want))
    return want, single


def _port_details(port, sr, reads, mer, forward, max_match, **kw):
    h = port.index_create(sr, 13, mer)
    a = port.aligner_create(h, forward=forward, max_match=max_match, **kw)
    try:
        return port_details(port, a, sr, reads)
    finally:
        port.aligner_destroy(a)
        port.index_destroy(h)


@pytest.mark.parametrize("unitigs", [False, True], ids=["plain", "forward_unitigs"])
def test_jf_aligner_details_with_max_match(tmpdir_session, tmp_path, port, unitigs):
    """Several batches (MR_BATCH_BASES) on two streams per GPU (MR_STREAMS=2)."""
    info = gen_synth(os.path.join(tmpdir_session, "details_mm"), 200000, coverage=4, read_len=4000, seed=13, repeat_frac=0.2)
    cmd = [JFA, "-s", "1M", "-m", "15", "--max-match", "-r", info["sr"], "-p", info["reads"]]
    if unitigs:
        cmd += ["-f", "-l", info["unitigs_len"], "-k", "41"]
    env = dict(os.environ, MR_BATCH_BASES="150000", MR_STREAMS="2")
    want, single = _details_run(tmp_path, port, cmd, env, info["sr"], info["reads"], info["unitigs_len"] if unitigs else None,
                                15, 41, unitigs)
    assert len(want) > 500
    # some group lost hits to discards: its line has fewer hits than the same group's line without --max-match
    n_single = {tuple(l.split()[:2]): len(l.split()) for l in single}
    assert any(len(l.split()) < n_single[tuple(l.split()[:2])] for l in want)


@pytest.mark.parametrize("forward", [False, True])
def test_jf_aligner_details_with_max_match_on_the_reference_fixture(tmp_path, port, forward):
    """The reference's own aligner_output inputs (k = 17, --stretch-cap 200) with --max-match added."""
    sr, reads, ul = (os.path.join(GOLD, n) for n in ("test_super_reads.fa", "test_pacbio.fa", "test_unitigs_lengths"))
    cmd = [JFA, "-s", "10k", "-m", "17", "-r", sr, "-p", reads, "--stretch-cap", "200", "--max-match"]
    if forward:
        cmd += ["-l", ul, "-k", "65", "-f"]
    want, _ = _details_run(tmp_path, port, cmd, None, sr, reads, ul if forward else None, 17, 65 if forward else 0, forward,
                           stretch_cap=200.0)
    assert len(want) == 3
