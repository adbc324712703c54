"""GPU parity tests, stage by stage, through the C ABI (ctypes) against the oracle port -- and
against the compiled reference when oracle/_ref travelled to the box."""
import os

import numpy as np
import pytest

from oracle_lib import device_rows, gen_synth, oracle_rows, read_fasta

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]


@pytest.fixture(scope="module")
def ctx():
    import pacbio_b200 as pb
    c = pb.Context(0)
    yield c
    c.close()


def _queries(k, n, seed, sr_text_codes):
    rng = np.random.default_rng(seed)
    q = rng.integers(0, 4 ** k, size=n, dtype=np.uint64)
    pos = rng.integers(0, len(sr_text_codes) - k, size=n // 2)
    w = (4 ** np.arange(k - 1, -1, -1)).astype(np.uint64)
    for i, p in enumerate(pos):
        codes = sr_text_codes[p:p + k].astype(np.uint64)
        if i & 1:
            codes = 3 - codes[::-1]
        q[i] = int((codes * w).sum())
    return q


CASES = [
    dict(name="k15", genome=150000, coverage=3, read_len=4000, seed=31, repeat_frac=0.15, k=15, m=13, uk=41),
    dict(name="k17", genome=120000, coverage=3, read_len=5000, seed=32, repeat_frac=0.0, k=17, m=13, uk=41, error=0.12),
    dict(name="k19m10", genome=60000, coverage=4, read_len=3000, seed=33, repeat_frac=0.25, k=19, m=10, uk=31,
         mean_unitig=200, error=0.10),
    dict(name="k16", genome=80000, coverage=3, read_len=2500, seed=34, repeat_frac=0.1, k=16, m=12, uk=41),
]


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
    yield dict(cfg=c, info=info, sr=sr, ul=ul, idx=idx, hp=hp)
    idx.close()
    port.index_destroy(hp)


def test_index_matches_oracle(case, port):
    idx, hp, c = case["idx"], case["hp"], case["cfg"]
    assert np.array_equal(idx.sa(), port.sa(hp))
    assert np.array_equal(idx.counts(), port.counts(hp, c["m"]))


def test_saved_index_loads_identically(case, ctx, port, tmp_path):
    """mr_index_save / mr_index_load: the loaded index is the built one (SA, counts, lookups, checksum)."""
    import pacbio_b200 as pb
    idx, c, sr = case["idx"], case["cfg"], case["sr"]
    path = str(tmp_path / "index.bin")
    idx.save(path)
    ctx2 = pb.Context(0)
    try:
        back = pb.Index(ctx2, sr, c["m"], c["k"], load_from=path)
        assert back.checksum() == idx.checksum() != 0
        assert np.array_equal(back.sa(), idx.sa())
        assert np.array_equal(back.counts(), idx.counts())
        rng = np.random.default_rng(5)
        q = rng.integers(0, 4 ** c["k"], size=5000, dtype=np.uint64)
        q[:2500] = [int(x) for x in _text_kmers(case, 2500, c["k"])]
        a, b = idx.lookup(q), back.lookup(q)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and int(a[1].sum()) >= 2500
        back.close()
        # a truncated file and a file that is not an index are refused
        raw = open(path, "rb").read()
        open(path, "wb").write(raw[:len(raw) // 2])
        with pytest.raises(pb.MrError):
            pb.Index(ctx2, sr, c["m"], c["k"], load_from=path)
        open(path, "wb").write(b"not an index" * 100)
        with pytest.raises(pb.MrError):
            pb.Index(ctx2, sr, c["m"], c["k"], load_from=path)
    finally:
        ctx2.close()


def _text_kmers(case, n, k):
    _, seqs = read_fasta(case["info"]["sr"])
    b = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    codes = (((b >> 1) ^ (b >> 2)) & 3).astype(np.uint64)
    rng = np.random.default_rng(9)
    w = (4 ** np.arange(k - 1, -1, -1)).astype(np.uint64)
    starts = np.cumsum([0] + [len(s) for s in seqs])
    out = []
    while len(out) < n:
        s = int(rng.integers(0, len(seqs)))
        if len(seqs[s]) < k:
            continue
        p = int(starts[s] + rng.integers(0, len(seqs[s]) - k + 1))
        out.append(int((codes[p:p + k] * w).sum()))
    return out


def test_lookup_matches_oracle(case, port):
    idx, hp, c, sr = case["idx"], case["hp"], case["cfg"], case["sr"]
    _, seqs = read_fasta(case["info"]["sr"])
    b = np.frombuffer("".join(seqs).encode(), dtype=np.uint8)
    codes = ((b >> 1) ^ (b >> 2)) & 3
    q = _queries(c["k"], 20000, 7, codes)
    # k-mers that collide with the tail-short suffixes of the text (padded with A)
    k, n = c["k"], len(codes)
    extra = []
    for j in range(1, k - c["m"] + 1):
        v = 0
        for t in range(k):
            p = n - k + j + t
            v = (v << 2) | (int(codes[p]) if p < n else 0)
        extra.append(v)
    q = np.concatenate([q, np.array(extra, dtype=np.uint64)])
    gi, gn = idx.lookup(q)
    oi, on = port.search(hp, q)
    assert np.array_equal(gn, on)
    assert np.array_equal(gi, oi)
    assert int(gn.sum()) > 5000


@pytest.mark.parametrize("k", [15, 17, 19])
def test_lookup_at_scale_matches_reference_psa_search(ctx, port, tmpdir_session, k):
    """BASELINE.json configs[4] parity: mr_lookup_batch == PSA::search (mer_sa_imp.hpp:369-479, through the
    compiled reference's libref_tap.so when it travelled to the box, else the oracle port) on a 64 Mbp random
    text x 1e6 queries -- half sampled from the text (both strands), half uniform random -- at k = 15 / 17 / 19."""
    import pacbio_b200 as pb
    from oracle_lib import Ref, have_ref
    n, nq, m = 64_000_000, 1_000_000, 13
    fa = os.path.join(tmpdir_session, "lookup_scale.fa")
    rng = np.random.default_rng(4600)
    if not os.path.exists(fa):
        codes = rng.integers(0, 4, size=n, dtype=np.uint8)
        with open(fa, "wb") as f:                       # 16 sequences of 4 Mbp, one line each
            for i in range(16):
                f.write(b">%d\n" % i)
                f.write(np.frombuffer(b"ACGT", dtype=np.uint8)[codes[i * (n // 16):(i + 1) * (n // 16)]].tobytes())
                f.write(b"\n")
    sr = pb.SuperReads(fa)
    assert sr.n == n
    words = sr.text2bit
    qr = np.random.default_rng(4700 + k)
    pos = qr.integers(0, n - k, size=nq // 2).astype(np.int64)
    fwd = np.zeros(nq // 2, dtype=np.uint64)
    rc = np.zeros(nq // 2, dtype=np.uint64)
    for j in range(k):
        b = pos + j
        code = (words[b >> 5] >> (2 * (b & 31)).astype(np.uint64)) & np.uint64(3)
        fwd = (fwd << np.uint64(2)) | code
        rc = rc | ((np.uint64(3) - code) << np.uint64(2 * j))
    q = np.concatenate([np.where(np.arange(nq // 2) & 1, rc, fwd), qr.integers(0, 4 ** k, size=nq - nq // 2, dtype=np.uint64)])
    idx = ctx.index(sr, m, k)
    try:
        gi, gn = idx.lookup(q)
    finally:
        idx.close()
    checker = Ref() if have_ref() else port
    h = checker.index_create(fa, m, k, 16)
    try:
        oi, on = checker.search(h, q)
    finally:
        checker.index_destroy(h)
    assert np.array_equal(gn, on)
    assert np.array_equal(gi, oi)
    assert int((gn > 0).sum()) >= nq // 4           # every k-mer sampled on the text's own strand is found (the search is strand specific)


@pytest.mark.parametrize("forward,window", [(True, 1), (False, 1), (True, 3), (False, 2)])
def test_align_stages_match_oracle(case, ctx, port, forward, window):
    """hit lists, both chains and coords rows of every (read, super-read) pair against the oracle port; window > 1 is
    --window-size (lis_align.hpp:17-45,162-163: the mer predicate on the sum of the last `window` steps)"""
    import pacbio_b200 as pb
    c = case["cfg"]
    reads = pb.Reads(case["info"]["reads"])
    nreads = min(reads.nreads, 60)
    sub = reads.slice(0, nreads)
    # a read with an N run and a tiny read, to exercise the k-mer restart and the empty paths
    names, seqs = read_fasta(case["info"]["reads"])
    seqs = seqs[:nreads]
    s0 = seqs[0]
    seqs.append(s0[:700] + "NNNN" + s0[704:1500] + "n" + s0[1501:2400])
    seqs.append("ACGT")
    seqs.append("")
    _, srs = read_fasta(case["info"]["sr"])
    longest = max(srs, key=len)
    seqs.append(longest[:min(len(longest), 6000)])          # one chain of thousands of hits
    sub = pb.Reads(names=["r%d" % i for i in range(len(seqs))], seqs=seqs)
    uk = c["uk"] if forward else 0
    p = pb.default_params(unitigs_k=uk, run_graph=0, forward=int(forward), window_size=window)
    ctx.keep_taps(True)
    res = ctx.align(case["idx"], sub, p)
    ctx.keep_taps(False)
    # the same reads without taps: single-hit groups and groups of up to 8 hits then take their own kernels
    prod = ctx.align(case["idx"], sub, p)
    ap = port.aligner_create(case["hp"], unitigs_k=uk, forward=forward, window_size=window)
    total_coords = 0
    for r, s in enumerate(seqs):
        o = port.align_read(ap, s)
        rows = res.tap_groups[res.tap_groups[:, 0] == r]
        assert np.array_equal(rows[:, 1:], o["groups"]), "groups of read %d" % r
        # offsets / lis of this read: contiguous slices in group order
        first = int(np.flatnonzero(res.tap_groups[:, 0] == r)[0]) if len(rows) else 0
        off0 = int(res.tap_groups[:first, 2:4].sum())
        lis0 = int(res.tap_groups[:first, 4:6].sum())
        noff, nlis = int(o["groups"][:, 1:3].sum()), int(o["groups"][:, 3:5].sum())
        assert np.array_equal(res.tap_offsets[off0:off0 + noff], o["offsets"]), "hit lists of read %d" % r
        assert np.array_equal(res.tap_lis[lis0:lis0 + nlis], o["lis"]), "chains of read %d" % r
        want = oracle_rows(o)
        assert device_rows(res, r, len(s)) == want, "coords of read %d" % r
        assert device_rows(prod, r, len(s)) == want, "coords of read %d without taps" % r
        total_coords += len(want)
    assert total_coords > 20
    port.aligner_destroy(ap)


def test_packed_entry_point_gives_the_same_rows(case, ctx):
    """mr_align_batch (characters, packed on the device) == mr_align_batch_packed (packed on the host by mr_pack_reads)."""
    import pacbio_b200 as pb
    c = case["cfg"]
    reads = pb.Reads(case["info"]["reads"])
    p = pb.default_params(unitigs_k=c["uk"], run_graph=1)
    a, b = ctx.align(case["idx"], reads, p), ctx.align_packed(case["idx"], reads, p)
    assert a.ncoords == b.ncoords > 0 and np.array_equal(a.read_coords, b.read_coords)
    for f in ("rs", "re", "qs", "qe", "nb_mers", "sr", "use_bwd", "lpath", "lstart", "lprev", "component", "info_len"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert np.array_equal(a.stretch.view(np.uint64), b.stretch.view(np.uint64))
    for row in range(0, a.ncoords, 7):               # (a row's slice of kmers_info sits wherever its survivor slot put it)
        assert np.array_equal(a.info(row)[0], b.info(row)[0]) and np.array_equal(a.info(row)[1], b.info(row)[1])


def test_staged_batches_give_the_same_rows(case, ctx):
    """mr_stage_batch + mr_align_staged (copy of the next batch under the kernels of the current one) == mr_align_batch."""
    import pacbio_b200 as pb
    c = case["cfg"]
    reads = pb.Reads(case["info"]["reads"])
    p = pb.default_params(unitigs_k=c["uk"], run_graph=1)
    want = ctx.align(case["idx"], reads, p)
    s1 = ctx.stage(reads)
    s2 = ctx.stage(reads)                      # two batches in flight on the copy stream
    got1 = ctx.align_staged(case["idx"], s1, p)
    got2 = ctx.align_staged(case["idx"], s2, p)
    for got in (got1, got2):
        assert got.ncoords == want.ncoords and got.ncoords > 0
        for f in ("rs", "re", "qs", "qe", "nb_mers", "sr", "stretch", "offset", "avg_err", "lpath", "lprev", "component"):
            assert np.array_equal(getattr(got, f), getattr(want, f)), f
    s3 = ctx.stage(reads)                      # a staged batch that is never aligned can be dropped
    ctx.L.mr_staged_free(s3)


@pytest.mark.parametrize("max_count", [5000, 3])
def test_index_of_several_parts_gives_the_same_lists_and_rows(case, ctx, max_count, tmp_path):
    """A text of 2^32 bases or more is indexed as several parts (index.cuh); MR_INDEX_PART_BASES forces
    that on a small input.  Hit lists, chains, rows and graph must not depend on the cut -- including
    the list sizes the count filters see (k-mers straddling two super-reads at a cut, max-count on the
    sum over the parts)."""
    import pacbio_b200 as pb
    c = case["cfg"]
    sr = case["sr"]
    assert case["idx"].parts() == 1
    os.environ["MR_INDEX_PART_BASES"] = str(max(1024, int(sr.n / 3.3)))
    try:
        idx = ctx.index(sr, c["m"], c["k"], unitig_len=case["ul"])
    finally:
        del os.environ["MR_INDEX_PART_BASES"]
    try:
        assert idx.parts() in (3, 4)
        reads = pb.Reads(case["info"]["reads"])
        names, seqs = read_fasta(case["info"]["reads"])
        _, srs = read_fasta(case["info"]["sr"])
        # reads that are super-read junctions: their k-mers straddle two consecutive super-reads
        seqs = seqs[:80] + [srs[i][-200:] + srs[i + 1][:200] for i in range(0, len(srs) - 1, max(1, len(srs) // 40))]
        sub = pb.Reads(names=["r%d" % i for i in range(len(seqs))], seqs=seqs)
        p = pb.default_params(unitigs_k=c["uk"], run_graph=1)
        p.max_count = max_count
        out = []
        for ix in (case["idx"], idx):
            ctx.keep_taps(True)
            out.append(ctx.align(ix, sub, p))
            ctx.keep_taps(False)
        want, got = out
        assert want.ncoords > 20 or max_count < 10
        for f in ("tap_groups", "tap_offsets", "tap_lis"):
            assert np.array_equal(getattr(got, f), getattr(want, f)), f
        assert got.ncoords == want.ncoords
        for f in ("rs", "re", "qs", "qe", "nb_mers", "pb_cons", "sr_cons", "pb_cover", "sr_cover", "ql", "rn", "sr", "use_bwd",
                  "stretch", "offset", "avg_err", "info_len", "lpath", "lprev", "lstart", "lunitigs", "component"):
            assert np.array_equal(getattr(got, f), getattr(want, f)), f
        # what is defined for one suffix array only says so
        with pytest.raises(Exception):
            idx.sa()
        # an index of several parts goes through a file like any other
        path = str(tmp_path / "parts.bin")
        idx.save(path)
        back = pb.Index(ctx, sr, c["m"], c["k"], load_from=path)
        try:
            assert back.parts() == idx.parts() and back.checksum() == idx.checksum() != 0
            again = ctx.align(back, sub, p)
            assert again.ncoords == want.ncoords
            for f in ("rs", "re", "qs", "qe", "nb_mers", "ql", "sr", "stretch", "offset", "avg_err", "info_len", "lpath", "lprev", "component"):
                assert np.array_equal(getattr(again, f), getattr(want, f)), f
        finally:
            back.close()
    finally:
        idx.close()


def test_random_sector_ceiling_microkernel(ctx):
    """mr_selftest_random_gather (bench.py's roofline denominator) runs and reports a plausible figure."""
    import ctypes as C
    g = C.c_double()
    ctx.check(ctx.L.mr_selftest_random_gather(ctx.h, 256 << 20, 1 << 24, C.byref(g)))
    assert 50.0 < g.value < 20000.0, g.value


def test_shared_reciprocal_division_is_exact(ctx):
    """div_by_count (chain.cu) must equal IEEE x / n bit for bit: 2^30 random operands."""
    import ctypes as C
    L = ctx.L
    L.mr_selftest_division.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.POINTER(C.c_uint64)]
    for seed, max_n in ((1, 70000), (2, 1 << 20), (3, 40)):
        bad = C.c_uint64(123)
        ctx.check(L.mr_selftest_division(ctx.h, 1 << 28, seed, max_n, C.byref(bad)))
        assert bad.value == 0


def test_max_match_coords_match_oracle(case, ctx, port):
    """--max-match: every secondary row (coarse_aligner.cc:56-57) must match the oracle, doubles bit for bit."""
    import pacbio_b200 as pb
    c = case["cfg"]
    _, seqs = read_fasta(case["info"]["reads"])
    seqs = seqs[:30]
    # reads holding the same super-read segment twice: the second copy can only be reported as a
    # secondary match, after the first chain has been discarded
    _, srs = read_fasta(case["info"]["sr"])
    for s_ in [x for x in srs if len(x) > 2500][:6]:
        seqs.append(s_[100:1300] + "ACGTTGCA" + s_[100:1300] + s_[1300:2000])
    # an error-free copy of a long super-read slice: one chain of thousands of hits (the long-chain
    # finisher; a mis-compiled variant of it once hung on exactly this)
    longest = max(srs, key=len)
    seqs.append(longest[:min(len(longest), 6000)])
    n = len(seqs)
    sub = pb.Reads(names=["r%d" % i for i in range(n)], seqs=seqs)
    p = pb.default_params(unitigs_k=c["uk"], run_graph=0, max_match=1)
    res = ctx.align(case["idx"], sub, p)
    ap = port.aligner_create(case["hp"], unitigs_k=c["uk"], max_match=True)
    extra = 0
    for r in range(n):
        o = port.align_read(ap, seqs[r])
        rr = list(res.rows(r))
        assert device_rows(res, r, len(seqs[r])) == oracle_rows(o), "coords of read %d" % r
        extra += len(rr) - len(set(res.sr[rr].tolist()))
    assert extra > 0, "no secondary match was exercised"
    port.aligner_destroy(ap)
