"""Bulk BAM mode (nb_process_bam_bulk, `nimble --bulk`) restated in Python for the tests: the FASTQs a BAM without cell
barcodes stands for, and the pairs the device forms from it.

A record is (qname, flag, seq) with seq in BAM's letters "=ACMGRSVTWYHKDBN".  The FASTQ text of a REVERSE record is what
`samtools fastq` writes: reversed, with the IUPAC complement (a non-ACGT letter stays non-ACGT).  FASTQ mode reads every
non-ACGT letter as A, so the reads the device aligns are `fastq_mode(fastq_text(...))`; the tests hand the text itself to the
FASTQ driver, so that the two readings are checked against each other."""
import collections
import os

from oracle import bam_ref

Rec = collections.namedtuple("Rec", "qname flag seq")

PAIRED, REVERSE, READ1, READ2, SECONDARY, SUPPLEMENTARY = 0x1, 0x10, 0x40, 0x80, 0x100, 0x800
FLAG_REVCOMP_FASTQ = 4                     # NB_FLAG_REVCOMP_FASTQ
_IUPAC = str.maketrans("ACGTMRWSYKVHDBN=", "TGCAKYWSRMBDHVN=")


class Refused(Exception):
    """what nb_process_bam_bulk refuses (NB_ERR_UNSUPPORTED): a mixed file, a kept record without SEQ"""


def read_bam(path):
    return [Rec(r.qname, r.flag, r.seq) for r in bam_ref.read_bam(path)]


def kept(records):
    """(ordinal, record) of every record that is neither secondary nor supplementary"""
    out = []
    for i, r in enumerate(records):
        if r.flag & (SECONDARY | SUPPLEMENTARY):
            continue
        if not r.seq:
            raise Refused("record %d has no SEQ" % i)
        out.append((i, r))
    return out


def fastq_text(r):
    """the read as samtools fastq writes it"""
    return r.seq[::-1].translate(_IUPAC) if r.flag & REVERSE else r.seq


def fastq_mode(text):
    """DnaString::from_acgt_bytes, as the FASTQ driver reads a line"""
    return "".join(c if c in "ACGT" else "A" for c in text.upper())


def pairs(records):
    """-> (paired, [(ordinal of R1, ordinal of R2 or None)]) sorted by R1 ordinal; Refused as the device path refuses"""
    k = kept(records)
    with_1 = [i for i, r in k if r.flag & PAIRED]
    without = [i for i, r in k if not r.flag & PAIRED]
    if with_1 and without:
        raise Refused("record %d is paired and record %d is not" % (with_1[0], without[0]))
    if not with_1:
        return False, [(i, None) for i, _ in k]
    templates = collections.OrderedDict()
    for i, r in k:
        templates.setdefault(r.qname, []).append((i, r))
    out = []
    for members in templates.values():
        if len(members) != 2:
            continue
        r1 = [i for i, r in members if r.flag & (READ1 | READ2) == READ1]
        r2 = [i for i, r in members if r.flag & (READ1 | READ2) == READ2]
        if len(r1) == 1 and len(r2) == 1:
            out.append((r1[0], r2[0]))
    return True, sorted(out)


def dump_lines(records):
    """the lines of nb_bam_dump_pairs_bulk"""
    paired, ps = pairs(records)
    def f(r):
        return FLAG_REVCOMP_FASTQ if r.flag & REVERSE else 0
    lines = []
    for a, b in ps:
        ra = records[a]
        if paired:
            rb = records[b]
            lines.append("%d\t%d\t%d\t%d\t%d\t%d" % (a, b, len(ra.seq), len(rb.seq), f(ra), f(rb)))
        else:
            lines.append("%d\t-\t%d\t-\t%d\t-" % (a, len(ra.seq), f(ra)))
    return lines


def write_fastqs(records, directory, stem="bulk"):
    """The FASTQ(s) the BAM stands for, in R1-ordinal order -> [r1.fastq, r2.fastq] or [r.fastq]"""
    paired, ps = pairs(records)
    names = ["%s_r1.fastq" % stem, "%s_r2.fastq" % stem] if paired else ["%s_r.fastq" % stem]
    paths = [os.path.join(str(directory), n) for n in names]
    for side, path in enumerate(paths):
        with open(path, "w") as f:
            for p in ps:
                r = records[p[side]]
                t = fastq_text(r)
                f.write("@%s\n%s\n+\n%s\n" % (r.qname, t, "I" * len(t)))
    return paths
