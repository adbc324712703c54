"""Chaining and coords at the edges of every route of launch_chain (chain.cu) and kmers_info_kernel (align.cu).

The input is engineered, from a fixed seed: random super-reads with synthetic unitig paths, and reads cut from them
so that (read, super-read) groups land exactly on the size classes' edges:

* groups of 1 hit (the single-hit shortcut of classify_groups_kernel), 2 .. 8 hits (chain_tiny_kernel), c - 1 / c /
  c + 1 hits for every shared-memory tier cap c (chain_coords_smem_kernel), and more than 4096 (the global-memory
  kernel), each on the forward strand only, the backward strand only and split across both;
* chains of 1535 / 1536 / 1537 hits (finish_tile_kernel against finish_warp_kernel) and 2048 / 2049 (the end of the
  reciprocal table);
* stray front entries: q hits late in a super-read followed by a long run earlier in it, so that every hit of the
  run is inserted behind q list entries (q = 32 is the last depth chain_strand_smem appends runs at);
* enough groups of tiers 0, 1 and 5 to fill whole 32-chain warps of the coords kernels, with mixed chain lengths
  (the 16-pair tiles, the 8-hit pieces of kmers_info_kernel);
* shuffled tiny groups, reads with errors near the tier edges and reads across a super-read junction;
* unitig paths of 1, 2, 24 and 25 (kInfoLocal) and 40 unitigs, one with a unitig shorter than k_u - 1, one with an
  unknown unitig id and one super-read name that does not parse.

Segment lengths are calibrated with the oracle port, which gives every group's hit counts and chain lengths directly.
The CPU test checks that every edge is present; the GPU tests compare every row, bit for bit, with the oracle, with
parity taps on (hit lists and both chains too) and off (the routes production runs).
"""
import os

import numpy as np
import pytest

from oracle_lib import device_rows, oracle_rows

K, PSA_MIN, UK = 15, 13, 41
TIER_CAPS = (64, 256, 512, 768, 1024, 1536, 2048, 3072, 4096)
SIZES = sorted({1, 2, 3, 8, 9, 10, 6000} | {c + d for c in TIER_CAPS for d in (-1, 0, 1)})
CHAINS = (1535, 1536, 1537, 2048, 2049, 4100)
DEPTHS = (1, 31, 32, 33, 64)
DEPTH_HOSTS = {"tier 1": 160, "tier 8": 3500, "global": 4700}       # group sizes of the stray-entry reads
TILE_TIERS = {0: (9, 64), 1: (65, 256), 5: (1025, 1536)}
TILE_CHAINS = (1, 8, 9, 15, 16, 17, 31, 32, 33, 256, 257, 264)
PATH_LENGTHS = (1, 2, 24, 25, 40)
BASES = np.array(list("ACGT"))
COMP = str.maketrans("ACGT", "TGCA")


def _rc(s):
    return s.translate(COMP)[::-1]


def _tier(n):
    for t, c in enumerate(TIER_CAPS):
        if n <= c:
            return t
    return len(TIER_CAPS)


class _Builder:
    """Super-reads, unitig paths and calibrated reads (all choices from one seeded generator)."""

    def __init__(self, port, tmpdir, seed=20261020):
        self.rng = np.random.default_rng(seed)
        self.port = port
        self.dir = tmpdir
        self._super_reads()
        self.hp = port.index_create(self.sr_fa, PSA_MIN, K)
        port.set_unitigs_lengths(self.hp, self.ul)
        # accept-all filters: group sizes and chains do not depend on the filters, rows then exist for every group
        self.ap = port.aligner_create(self.hp, unitigs_k=UK, matching_mers=0.0, matching_bases=0.0)
        self.reads, self.kinds = [], []

    # ---- super-reads -------------------------------------------------------------------------------------------
    def _random(self, n):
        return "".join(BASES[self.rng.integers(0, 4, size=n)])

    def _path(self, length, n):
        """Unitig lengths of an n-unitig path spelling `length` bases with k_u - 1 overlaps."""
        if n == 1:
            return [length]
        cuts = np.sort(self.rng.choice(np.arange(1, length), size=n - 1, replace=False))
        adv = np.diff(np.concatenate([[0], cuts, [length]]))
        return [int(adv[0])] + [int(a) + UK - 1 for a in adv[1:]]

    def _super_reads(self):
        rng = self.rng
        npaths = list(PATH_LENGTHS) + ["short unitig", "unknown id", "no name"] + \
            [int(x) for x in rng.integers(2, 25, size=52)]
        seqs = [self._random(int(rng.integers(7000, 12001))) for _ in npaths] + \
               [self._random(int(rng.integers(20, 121))) for _ in range(10)]
        npaths += [int(rng.integers(1, 3)) if len(s) >= 2 * UK else 1 for s in seqs[len(npaths):]]
        names, ul, self.path_of = [], [], []
        for s, npath in zip(seqs, npaths):
            n = npath if isinstance(npath, int) else 6
            lens = self._path(len(s), n)
            if npath == "short unitig":                 # a unitig shorter than k_u - 1, its neighbour takes up the slack
                lens[2], lens[3] = UK - 11, lens[3] + lens[2] - (UK - 11)
            ids = list(range(len(ul), len(ul) + n))
            ul += lens
            if npath == "unknown id":
                ids[0] = 10 ** 6
            name = "_".join("%d%s" % (i, "FR"[int(rng.integers(0, 2))]) for i in ids)
            if npath == "no name":
                name = "noname"
            names.append(name)
            self.path_of.append(npath)
        self.seqs, self.names = seqs, names
        self.ul = np.array(ul, dtype=np.int64)
        self.long = [i for i, s in enumerate(seqs) if len(s) >= 7000]
        self.short = [i for i, s in enumerate(seqs) if len(s) < 7000]
        self.sr_fa = os.path.join(self.dir, "edges.superreads.fa")
        self.ul_txt = os.path.join(self.dir, "edges.unitigs_len.txt")
        with open(self.sr_fa, "w") as f:
            for n, s in zip(names, seqs):
                f.write(">%s\n%s\n" % (n, s))
        with open(self.ul_txt, "w") as f:
            for i, x in enumerate(ul):
                f.write("%d %d\n" % (i, x))

    # ---- reads -------------------------------------------------------------------------------------------------
    def junk(self, n, before=None, after=None):
        """n random bases; the first differs from `before`'s continuation base, the last from `after`'s preceding
        base, so that no k-mer across a segment's end matches by a lucky junk base."""
        j = list(self._random(n))
        if n and before is not None:
            while j[0] == before:
                j[0] = BASES[self.rng.integers(0, 4)]
        if n and after is not None:
            while j[-1] == after or (n == 1 and j[0] == before):
                j[-1] = BASES[self.rng.integers(0, 4)]
        return "".join(j)

    def piece(self, sr, start, length, bwd):
        """(text, base expected right before it in the read, base expected right after it)."""
        s = self.seqs[sr]
        t = s[start:start + length]
        prev = s[start - 1] if start > 0 else None
        nxt = s[start + length] if start + length < len(s) else None
        if bwd:
            return _rc(t), (nxt.translate(COMP) if nxt else None), (prev.translate(COMP) if prev else None)
        return t, prev, nxt

    def assemble(self, pieces, gap=(3, 12)):
        """pieces: (sr, start, length, bwd); random junk around and between them."""
        out, last_next = [], None
        for sr, start, length, bwd in pieces:
            t, before, after = self.piece(sr, start, length, bwd)
            out.append(self.junk(int(self.rng.integers(*gap)), before=last_next, after=before))
            out.append(t)
            last_next = after
        out.append(self.junk(int(self.rng.integers(*gap)), before=last_next))
        return "".join(out)

    def group(self, seq, sr):
        o = self.port.align_read(self.ap, seq)
        row = o["groups"][o["groups"][:, 0] == sr]
        return tuple(int(x) for x in row[0, 1:]) if len(row) else (0, 0, 0, 0)

    def calibrate(self, make, target, metric, guess):
        """make(L) -> read; finds L with metric(read) == target (hits grow by one per base away from the edges)."""
        L, seen = max(1, guess), {}
        for _ in range(12):
            if L in seen:
                break
            seq = make(L)
            got = metric(seq)
            seen[L] = (got, seq)
            if got == target:
                return seq, L
            L = max(1, L + target - got)
        for L in sorted(seen, key=lambda x: abs(seen[x][0] - target)):      # local search around the best
            for d in (-3, -2, -1, 1, 2, 3):
                seq = make(L + d)
                if metric(seq) == target:
                    return seq, L + d
            break
        raise AssertionError("could not calibrate to %d (got %s)" % (target, sorted(v[0] for v in seen.values())))

    def pick(self, need, pool=None):
        pool = self.long if pool is None else pool
        ok = [i for i in pool if len(self.seqs[i]) >= need + 40]
        return ok[int(self.rng.integers(0, len(ok)))]

    def add(self, seq, kind):
        self.reads.append(seq)
        self.kinds.append(kind)

    @staticmethod
    def retry(fn, what, tries=8):
        """fn() -> read, or None when a check after the calibration fails (a chance hit elsewhere); each try draws
        a new super-read and position."""
        for _ in range(tries):
            try:
                out = fn()
            except AssertionError:
                continue
            if out is not None:
                return out
        raise AssertionError("no read for %s" % (what,))

    def sizes(self):
        for n in SIZES:
            for mode in ("fwd", "bwd", "split"):
                if mode == "split" and n == 1:
                    continue
                self.add(self.retry(lambda: self._size(n, mode), (n, mode)), ("size", n, mode))

    def _size(self, n, mode):
        sr = self.pick(n + 200)
        ls = len(self.seqs[sr])
        if mode != "split":
            st = int(self.rng.integers(1, ls - n - 60))
            seq, _ = self.calibrate(lambda L: self.assemble([(sr, st, L, mode == "bwd")]), n,
                                    lambda s: sum(self.group(s, sr)[:2]), n + 14)
            g = self.group(seq, sr)
            return seq if (g[1] if mode == "fwd" else g[0]) == 0 else None
        # the backward piece from the end of the super-read, the forward one from its start: n - 1 + 1, or 2n/3 + n/3
        nb = 1 if n < 64 or n % 2 else n // 3
        _, lb = self.calibrate(lambda L: self.assemble([(sr, 5, n - nb + 14, False), (sr, ls - L - 2, L, True)]),
                               nb, lambda s: self.group(s, sr)[1], nb + 14)
        seq, _ = self.calibrate(lambda L: self.assemble([(sr, 5, L, False), (sr, ls - lb - 2, lb, True)]),
                                n, lambda s: sum(self.group(s, sr)[:2]), n - nb + 14)
        return seq if self.group(seq, sr)[1] == nb else None

    def chains(self):
        for n in CHAINS:
            for bwd in (False, True):
                self.add(self.retry(lambda: self._chain(n, bwd), (n, bwd)), ("chain", n, bwd))

    def _chain(self, n, bwd):
        sr = self.pick(n + 200)
        st = int(self.rng.integers(1, len(self.seqs[sr]) - n - 60))
        seq, _ = self.calibrate(lambda L: self.assemble([(sr, st, L, bwd)]), n,
                                lambda s: max(self.group(s, sr)[2:]), n + 14)
        return seq

    def strays(self):
        for host, size in DEPTH_HOSTS.items():
            for q in DEPTHS:
                for bwd in (False, True):
                    self.add(self.retry(lambda: self._stray(q, size, bwd), (q, host, bwd)), ("stray", q, host))

    def _stray(self, q, size, bwd):
        """q hits from late in the super-read (early, on the backward strand) ahead of a long run from earlier."""
        sr = self.pick(size + 400)
        ls = len(self.seqs[sr])
        late = ls - q - 60 if not bwd else 30             # super-read offsets above every offset of the run
        run0 = 20 if not bwd else ls - size - 60

        def make(L, lq):
            return self.assemble([(sr, late, lq, bwd), (sr, run0, L, bwd)])
        depth = lambda s: _depth(self.port.align_read(self.ap, s), sr, bwd)
        _, lq = self.calibrate(lambda L: make(size - q + 14, L), q, depth, q + 14)
        seq, _ = self.calibrate(lambda L: make(L, lq), size, lambda s: sum(self.group(s, sr)[:2]), size - q + 14)
        return seq if depth(seq) == q else None

    def tiles(self):
        """Groups of tiers 0, 1, 5: a chain of c hits on one strand, single k-mers (a chain of 1) on the other."""
        for tier, (lo, hi) in TILE_TIERS.items():
            wanted = [c for c in TILE_CHAINS if c <= hi] + [0] * 4
            for j in range(80):
                c = wanted[j % len(wanted)] or int(self.rng.integers(1, hi + 1))
                n = int(self.rng.integers(max(lo, c), hi + 1))
                seq = self.retry(lambda: self._tile(n, c, bool(j & 1)), (tier, n, c))
                self.add(seq, ("tile", tier, c))

    def _tile(self, n, c, bwd):
        rng = self.rng
        paths = [i for i in self.long if isinstance(self.path_of[i], int) and 2 <= self.path_of[i] <= 24]
        sr = self.pick(c + 3 * (n - c) + 200, paths)
        ls = len(self.seqs[sr])
        st = int(rng.integers(1, max(2, ls - c - 3 * (n - c) - 100)))
        # the noise, one k-mer per piece on the other strand, ordered so that it never chains: forward hits with
        # super-read offsets decreasing along the read, backward hits with increasing positions
        # (a k-mer found twice in the text falls to the 99 % list-size cut, so the count is adjusted after a try)
        pool, m = rng.permutation(np.arange(st + c + 40, ls - K - 2)), n - c
        for _ in range(4):
            pos = np.sort(pool[:m])
            noise = [(sr, int(p), K, not bwd) for p in (pos[::-1] if bwd else pos)]
            make = lambda L: self.assemble([(sr, st, L, bwd)] + noise, gap=(2, 6))
            seq, _ = self.calibrate(make, c, lambda s: self.group(s, sr)[3 if bwd else 2], c + 14)
            g = self.group(seq, sr)
            if sum(g[:2]) == n and g[2 if bwd else 3] <= 1:
                return seq
            m += n - sum(g[:2])
        return None

    def tiny(self, count=330):
        """2 .. 8 hits in pieces of one or two k-mers of one super-read, shuffled, on random strands, in random junk."""
        rng = self.rng
        for _ in range(count):
            sr = self.pick(400)
            w0 = int(rng.integers(1, len(self.seqs[sr]) - 400))
            strand = bool(rng.integers(0, 2))
            pieces, left = [], int(rng.integers(2, 9))
            while left:
                nk = 2 if left >= 2 and rng.random() < 0.4 else 1
                pieces.append((sr, w0 + int(rng.integers(0, 300)), K + nk - 1, strand if rng.random() < 0.8 else not strand))
                left -= nk
            order = rng.permutation(len(pieces))
            self.add(self.assemble([pieces[i] for i in order], gap=(1, 40)), ("tiny",))

    def errors(self, count=54):
        """Reads with ~10 % substitutions and indels, calibrated to group sizes at the tier edges."""
        rng = self.rng
        targets = [c + d for c in (64, 256, 512, 768, 1024, 1536) for d in (-1, 0, 1)]
        for j in range(count):
            n = targets[j % len(targets)]
            sr = self.pick(int(n * 6.5) + 200)
            s = self.seqs[sr]
            st = int(rng.integers(1, 100))
            mut = []
            for ch in s[st:]:
                r = rng.random()
                if r < 0.06:
                    mut.append(BASES[(int("ACGT".index(ch)) + int(rng.integers(1, 4))) % 4])
                elif r < 0.08:
                    continue
                elif r < 0.10:
                    mut.append(ch + BASES[rng.integers(0, 4)])
                else:
                    mut.append(ch)
            text = "".join(mut)
            if j % 2:
                text = _rc(text)
            lo, hi = 1, len(text)
            size = lambda L: sum(self.group(text[:L] if not j % 2 else text[-L:], sr)[:2])
            while lo < hi:                                   # smallest prefix with at least n hits
                mid = (lo + hi) // 2
                if size(mid) >= n:
                    hi = mid
                else:
                    lo = mid + 1
            self.add(text[:lo] if not j % 2 else text[-lo:], ("errors", n))

    def junctions(self):
        for i in self.long[5:15]:
            if i + 1 < len(self.seqs):
                self.add(self.seqs[i][-150:] + self.seqs[i + 1][:150], ("junction",))

    def short_super_reads(self):
        for i in self.short:
            s = self.seqs[i]
            self.add(self.junk(30) + s + self.junk(30), ("short super-read",))
            self.add(self.junk(20) + _rc(s) + self.junk(40), ("short super-read",))

    def build(self):
        self.sizes()
        self.chains()
        self.strays()
        self.tiles()
        self.tiny()
        self.errors()
        self.junctions()
        self.short_super_reads()
        return self


def _depth(o, sr, bwd):
    """Stray depth of the group (read, sr) on one strand: the number of leading hits, in read order, whose
    super-read offsets all exceed every offset of the hits after them (0: none)."""
    g = o["groups"]
    idx = np.flatnonzero(g[:, 0] == sr)
    if not len(idx):
        return 0
    i = int(idx[0])
    off0 = int(g[:i, 1:3].sum())
    nf, nb = int(g[i, 1]), int(g[i, 2])
    sr_off = o["offsets"][off0 + (nf if bwd else 0):off0 + (nf + nb if bwd else nf), 1].astype(np.int64)
    if len(sr_off) < 2:
        return 0
    head_min = np.minimum.accumulate(sr_off)[:-1]
    tail_max = np.maximum.accumulate(sr_off[::-1])[::-1][1:]
    cut = np.flatnonzero(head_min > tail_max)
    return int(cut[-1]) + 1 if len(cut) else 0


@pytest.fixture(scope="module")
def edges(port, tmpdir_session):
    d = os.path.join(tmpdir_session, "chain_edges")
    os.makedirs(d, exist_ok=True)
    b = _Builder(port, d).build()
    yield b
    port.aligner_destroy(b.ap)
    port.index_destroy(b.hp)


def _coverage(b):
    """What the input holds, from the oracle port alone (accept-all filters)."""
    cov = dict(size={}, chain=set(), depth=set(), tile={t: 0 for t in TILE_TIERS}, tile_chain={t: set() for t in TILE_TIERS},
               tiny=0, path_rows={}, junction=0, rows=0)
    for seq, kind in zip(b.reads, b.kinds):
        o = b.port.align_read(b.ap, seq)
        g = o["groups"]
        cov["rows"] += len(o["cint"])
        for sr, nf, nb, lf, lb in g.tolist():
            n = nf + nb
            mode = "split" if nf and nb else ("fwd" if nf else "bwd")
            cov["size"].setdefault(n, set()).add(mode)
            cov["chain"].add(max(lf, lb))
            if 2 <= n <= 8 and kind[0] == "tiny":
                cov["tiny"] += 1
        gi = g[np.argmax(g[:, 1] + g[:, 2])] if len(g) else None        # the group the read was built for
        if kind[0] == "stray":
            q = _depth(o, int(gi[0]), gi[2] > gi[1])
            if _tier(int(gi[1] + gi[2])) == {"tier 1": 1, "tier 8": 8, "global": 9}[kind[2]]:
                cov["depth"].add((q, kind[2]))
        if kind[0] == "tile":
            if _tier(int(gi[1] + gi[2])) == kind[1]:
                cov["tile"][kind[1]] += 1
                cov["tile_chain"][kind[1]].add(int(max(gi[3], gi[4])))
        if kind[0] == "junction":
            # the k-mers across the junction are in the text but in no super-read: they form no group
            s = seq
            w = (4 ** np.arange(K - 1, -1, -1)).astype(np.uint64)
            codes = np.array(["ACGT".index(ch) for ch in s], dtype=np.uint64)
            mers = np.array([int((codes[i:i + K] * w).sum()) for i in range(150 - K + 1, 150)], dtype=np.uint64)
            _, found = b.port.search(b.hp, mers)
            cov["junction"] += int((found > 0).sum())
        for j, row in enumerate(o["cint"]):
            path = b.path_of[int(row[12])]
            ilen = int(o["info_off"][j + 1] - o["info_off"][j])
            cov["path_rows"].setdefault(path, [0, 0])[ilen > 0] += 1
    return cov


def test_engineered_input_reaches_every_edge(edges):
    """The input (built with the oracle port alone) reaches every edge the GPU tests rely on."""
    cov = _coverage(edges)
    lines = ["group size    strands"]
    lines += ["%10d    %s" % (n, ",".join(sorted(cov["size"].get(n, ())))) for n in SIZES]
    lines.append("chain lengths: %s" % sorted(c for c in cov["chain"] if c in set(CHAINS) | set(TILE_CHAINS) or c > 4096))
    lines.append("stray depths: %s" % sorted(cov["depth"]))
    lines.append("tile groups per tier: %s; chain lengths per tier: %s" % (cov["tile"], {t: sorted(v) for t, v in cov["tile_chain"].items()}))
    lines.append("tiny groups: %d; junction k-mers found in the text: %d; rows: %d" % (cov["tiny"], cov["junction"], cov["rows"]))
    lines.append("rows per unitig path (without info, with info): %s" % cov["path_rows"])
    print("\n".join(lines))
    for n in SIZES:
        want = {"fwd", "bwd"} | ({"split"} if n > 1 else set())
        assert want <= cov["size"].get(n, set()), "group size %d: %s" % (n, cov["size"].get(n))
    for c in CHAINS + TILE_CHAINS:
        assert c in cov["chain"], "chain of %d hits" % c
    for q in DEPTHS:
        for host in DEPTH_HOSTS:
            assert (q, host) in cov["depth"], "stray depth %d in a %s group" % (q, host)
    for t in TILE_TIERS:
        assert cov["tile"][t] >= 70, "tier %d: %d groups" % (t, cov["tile"][t])
    for t, want in ((0, (1, 15, 16, 17, 31, 32, 33, 8, 9)), (1, (1, 16, 33, 256)), (5, (1, 16, 256, 257, 264))):
        assert set(want) <= cov["tile_chain"][t], (t, sorted(cov["tile_chain"][t]))
    assert cov["tiny"] >= 300
    assert cov["junction"] > 0
    pr = cov["path_rows"]
    for n in (1, 2, 24, 25, 40, "short unitig"):
        assert pr.get(n, [0, 0])[1] > 0, "rows with kmers_info on a path of %s unitigs" % n
    assert pr.get("unknown id", [0, 0])[0] > 0                  # rows whose walk reaches the unknown unitig
    assert pr.get("no name", [0, 0])[0] > 0 and pr["no name"][1] == 0


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
ACCEPT_ALL = dict(matching_mers=0.0, matching_bases=0.0)
PARAM_SETS = {
    "A": dict(forward=1, unitigs_k=UK),
    "B": dict(forward=1, unitigs_k=UK, **ACCEPT_ALL),
    "C": dict(forward=0, unitigs_k=0, **ACCEPT_ALL),
    "D": dict(forward=1, unitigs_k=UK, window_size=2, **ACCEPT_ALL),
    "E": dict(forward=1, unitigs_k=UK, max_match=1, **ACCEPT_ALL),
}
RUNS = [(p, t) for p in "ABCD" for t in (True, False)] + [("E", False)]


def _subset(edges, pset):
    """Reads of a parameter set.  --max-match with accept-all filters makes a row of every noise hit of the tier-5
    tile groups, each after a chaining of the whole remaining group: quadratic, so E leaves those reads out."""
    if pset == "E":
        return [r for r, k in enumerate(edges.kinds) if k[:2] != ("tile", 5)]
    return list(range(len(edges.reads)))


@pytest.fixture(scope="module")
def gpu(edges):
    import pacbio_b200 as pb
    from oracle_lib import Ref, have_ref
    ctx = pb.Context(0)
    sr = pb.SuperReads(edges.sr_fa)
    idx = ctx.index(sr, PSA_MIN, K, unitig_len=edges.ul)
    checker = Ref() if have_ref() else edges.port
    hc = checker.index_create(edges.sr_fa, PSA_MIN, K)
    checker.set_unitigs_lengths(hc, edges.ul)
    state = dict(ctx=ctx, idx=idx, checker=checker, hc=hc, oracle={}, runs={})
    yield state
    checker.index_destroy(hc)
    idx.close()
    ctx.close()


def _oracle(gpu, edges, pset):
    if pset not in gpu["oracle"]:
        kw = dict(PARAM_SETS[pset])
        ap = gpu["checker"].aligner_create(gpu["hc"], unitigs_k=kw.pop("unitigs_k"), forward=bool(kw.pop("forward")),
                                           window_size=kw.pop("window_size", 1), max_match=bool(kw.pop("max_match", 0)),
                                           **kw)
        try:
            gpu["oracle"][pset] = [gpu["checker"].align_read(ap, edges.reads[r]) for r in _subset(edges, pset)]
        finally:
            gpu["checker"].aligner_destroy(ap)
    return gpu["oracle"][pset]


def _run(gpu, edges, pset, taps):
    import pacbio_b200 as pb
    if (pset, taps) not in gpu["runs"]:
        ctx = gpu["ctx"]
        sub = _subset(edges, pset)
        reads = pb.Reads(names=["r%d" % r for r in sub], seqs=[edges.reads[r] for r in sub])
        p = pb.default_params(run_graph=0, **PARAM_SETS[pset])
        ctx.keep_taps(taps)
        try:
            gpu["runs"][(pset, taps)] = ctx.align(gpu["idx"], reads, p)
        finally:
            ctx.keep_taps(False)
    return gpu["runs"][(pset, taps)]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("pset,taps", RUNS, ids=["%s-%s" % (p, "taps" if t else "notaps") for p, t in RUNS])
def test_chain_edges_match_oracle(edges, gpu, pset, taps):
    """Every row of every read equals the oracle's (integers exact, doubles bit for bit, kmers_info / bases_info);
    with taps on, the hit lists and both chains of every group too."""
    res = _run(gpu, edges, pset, taps)
    want = _oracle(gpu, edges, pset)
    sub = _subset(edges, pset)
    nrows = 0
    for r, (e, o) in enumerate(zip(sub, want)):
        s, what = edges.reads[e], "read %d %s" % (e, edges.kinds[e])
        if taps:
            sel = res.tap_groups[:, 0] == r
            rows = res.tap_groups[sel]
            assert np.array_equal(rows[:, 1:], o["groups"]), "groups of " + what
            first = int(np.flatnonzero(sel)[0]) if len(rows) else 0
            off0, lis0 = int(res.tap_groups[:first, 2:4].sum()), int(res.tap_groups[:first, 4:6].sum())
            noff, nlis = int(o["groups"][:, 1:3].sum()), int(o["groups"][:, 3:5].sum())
            assert np.array_equal(res.tap_offsets[off0:off0 + noff], o["offsets"]), "hit lists of " + what
            assert np.array_equal(res.tap_lis[lis0:lis0 + nlis], o["lis"]), "chains of " + what
        got = device_rows(res, r, len(s))
        assert got == oracle_rows(o), "coords of " + what
        nrows += len(got)
    assert nrows > len(sub) // 2
    if taps:
        sizes = set((res.tap_groups[:, 2] + res.tap_groups[:, 3]).tolist())
        assert set(SIZES) <= sizes, sorted(set(SIZES) - sizes)
    if pset != "A":                                   # accept-all filters: every group has its row
        assert {1537, 2049} <= set(res.nb_mers.tolist())
    if not taps and (pset, True) in gpu["runs"]:
        other = gpu["runs"][(pset, True)]
        assert all(device_rows(other, r, len(edges.reads[e])) == device_rows(res, r, len(edges.reads[e]))
                   for r, e in enumerate(sub)), "rows differ with and without taps"
