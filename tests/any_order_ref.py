"""The scopes of BAM mode in any record order (nb_process_bam_cells_any_order), stated on top of the CPU oracle of the grouped
reader (oracle/bam_ref.py) for the tests.  The oracle's readers are used as they are; the only addition is the record's file
ordinal on every item, so that the device's scopes can be compared record for record."""
from oracle import bam_ref


def read_bam(path):
    """bam_ref.read_bam with `ordinal` = the record's position in file order (Record.clone copies it)"""
    recs = bam_ref.read_bam(path)
    for i, r in enumerate(recs):
        r.ordinal = i
    return recs


class _OrdinalUMIReader(bam_ref.UMIReader):
    """bam_ref.UMIReader.next (src/parse/bam.rs:100-253) with the record's ordinal kept on each item"""

    def next(self):
        self.cur, self.nxt = self.nxt, []
        self.cur_key, self.nxt_key = self.nxt_key, ""
        while True:
            r = self.rd.next()
            if r is None:
                return True
            umi = bam_ref.SortedBamReader.umi_of(r)
            cb = r.aux_string("CB")
            if cb is None:
                raise RuntimeError("Error Read without cell barcode, cannot excise read-mate.")
            key = umi + cb[:-2]
            if self.cur_key == "":
                self.cur_key = key
            seq, qual, fields = bam_ref.record_fields(r)
            item = dict(seq=seq, qual=qual, f=fields, umi=umi, cb=cb[:-2], ordinal=getattr(r, "ordinal", None))
            if self.cur_key == key:
                self.cur.append(item)
            else:
                self.nxt.append(item); self.nxt_key = key
                return False


def _groups_of(records):
    """bam_ref.groups_of (src/process/bam.rs:157-180) over _OrdinalUMIReader"""
    rd = _OrdinalUMIReader(records, False)
    out = []; has_aligned = False
    while True:
        final = rd.next()
        if final and has_aligned:
            break
        out.append(list(rd.cur))
        has_aligned = True
        if final:
            break
    return out


def groups_any_order(records):
    """Stated literally: the records that fill_buffer keeps, stably sorted by (UMI, CB), followed by one scope with a UMI no
    record has, through the grouped reader; the sentinel's group is dropped.  Items carry the record's `ordinal`."""
    kept = []
    for r in records:
        if r.aux_string("CB") is None:
            continue
        umi = bam_ref.SortedBamReader.umi_of(r)
        if umi == "AAAAAAAAAA":
            continue
        kept.append(r)
    if not kept:
        return []
    kept.sort(key=lambda r: (bam_ref.SortedBamReader.umi_of(r), r.aux_string("CB")))
    s = kept[-1].clone()
    s.qname, s.flag, s.ordinal = "\0sentinel", 0, None
    s.aux = {"CB": ("Z", "~sentinel-1"), "UB": ("Z", "~" * (1 + max(len(bam_ref.SortedBamReader.umi_of(r)) for r in kept)))}
    groups = _groups_of(kept + [s])
    return [g for g in groups if g and g[0]["f"][0] != "\0sentinel"]
