"""The reference's jf_aligner --details printer (jf_aligner.cc:72-108) restated over the oracle port's per-read taps
(TEST INFRASTRUCTURE, never imported by the product).  The port's align_read returns every (read, super-read) group's
two hit lists and two chains in the state the reference prints them in: after the chaining, and with max_match after
the last discard of the loop in coarse_aligner.cc:42-60.  tests/test_details_cpu.py pins the printer to the
reference's own details_*_expected goldens."""
from oracle_lib import read_fasta


def super_read_names(sr_fasta):
    """Names of the super-reads in the port's index order: the whole header line after '>', sequences without bases
    skipped (superread_parser.cc:12-46, as oracle/port restates it)."""
    names, name, has_bases = [], None, False
    with open(sr_fasta) as f:
        for line in f:
            line = line.rstrip("\n")
            if line.startswith(">"):
                if name is not None and has_bases:
                    names.append(name)
                name, has_bases = line[1:], False
            elif line:
                has_bases = True
    if name is not None and has_bases:
        names.append(name)
    return names


def details_lines(read_name, taps, sr_names):
    """One line per group of one read: read name, super-read name, the hits of both lists merged by read offset (the
    forward hit first on equal offsets), those of the strictly longer list's chain in brackets."""
    out, off, li = [], 0, 0
    for sr, nf, nb, lf, lb in taps["groups"].tolist():
        fwd, bwd = taps["offsets"][off:off + nf].tolist(), taps["offsets"][off + nf:off + nf + nb].tolist()
        fwd_align = lf > lb
        chain = taps["lis"][li:li + lf].tolist() if fwd_align else taps["lis"][li + lf:li + lf + lb].tolist()
        off, li = off + nf + nb, li + lf + lb
        parts, fi, bi, c = [read_name, sr_names[sr]], 0, 0, 0
        while fi < nf or bi < nb:
            take_fwd = bi == nb or (fi < nf and fwd[fi][0] <= bwd[bi][0])
            (pb, so), i = (fwd[fi], fi) if take_fwd else (bwd[bi], bi)
            fi, bi = (fi + 1, bi) if take_fwd else (fi, bi + 1)
            in_chain = take_fwd == fwd_align and c < len(chain) and chain[c] == i
            c += in_chain
            parts.append(("[%d:%d]" if in_chain else "%d:%d") % (pb, so))
        out.append(" ".join(parts))
    return out


def port_details(port, aligner, sr_fasta, reads_fasta):
    """The lines jf_aligner --details writes for every read of reads_fasta, with the port aligner's parameters."""
    sr_names = super_read_names(sr_fasta)
    names, seqs = read_fasta(reads_fasta)
    out = []
    for name, seq in zip(names, seqs):
        out += details_lines(name, port.align_read(aligner, seq), sr_names)
    return out
