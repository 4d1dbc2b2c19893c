"""Compares extracted signature columns with the reference's candidate tuple lists (multisets)."""
import collections
import hashlib

from cutesv_b200 import packing


def digest_ins_seqs(cand):
    """The candidate dict with every INS sequence (tuple field 3) replaced by a 64-bit SHA-256 prefix: keeps stored
    goldens small while the comparison still covers the sequence content."""
    out = dict(cand)
    out["INS"] = [tuple(t[:3]) + ("sha256:" + hashlib.sha256(t[3].encode()).hexdigest()[:16],) + tuple(t[4:]) for t in cand["INS"]]
    return out


def tuples_from_columns(ex, chrom_names, read_names, query_of, cigar_of=None, merge=(10, 100)):
    """ex: dict(sigs, piece_off, piece_cnt, pieces, rows) -> the reference's tuple shapes.
    cigar_of(rec) -> (uint32 CIGAR array, reference_start) and merge = (min_siglength, merge_ins_threshold) are only needed
    for signatures that merged more insertions than the device buffers (piece flag 2)."""
    out = {k: [] for k in ("DEL", "INS", "DUP", "INV", "TRA")}
    s = ex["sigs"]["DEL"]
    for i in range(len(s["chrom"])):
        out["DEL"].append((int(s["a"][i]), int(s["b"][i]), read_names[int(s["read_id"][i])], "DEL", chrom_names[int(s["chrom"][i])]))
    s = ex["sigs"]["INS"]
    for i in range(len(s["chrom"])):
        a = int(s["a"][i])
        seq = packing.ins_sequence(ex["pieces"], int(ex["piece_off"][i]), int(ex["piece_cnt"][i]), query_of, cigar_of, merge)
        assert len(seq) == int(s["c"][i]), ("seq_len column", len(seq), int(s["c"][i]))
        out["INS"].append((a / 2, int(s["b"][i]), read_names[int(s["read_id"][i])], seq, "INS", chrom_names[int(s["chrom"][i])]))
    s = ex["sigs"]["DUP"]
    for i in range(len(s["chrom"])):
        out["DUP"].append((int(s["a"][i]), int(s["b"][i]), read_names[int(s["read_id"][i])], "DUP", chrom_names[int(s["chrom"][i])]))
    s = ex["sigs"]["INV"]
    for i in range(len(s["chrom"])):
        out["INV"].append(("++" if int(s["c"][i]) == 0 else "--", int(s["a"][i]), int(s["b"][i]), read_names[int(s["read_id"][i])], "INV",
                           chrom_names[int(s["chrom"][i])]))
    s = ex["sigs"]["TRA"]
    for i in range(len(s["chrom"])):
        c = int(s["c"][i])
        out["TRA"].append(("ABCD"[c & 3], int(s["a"][i]), chrom_names[c >> 2], int(s["b"][i]), read_names[int(s["read_id"][i])], "TRA",
                           chrom_names[int(s["chrom"][i])]))
    r = ex["rows"]
    rows = [(int(r["start"][i]), int(r["end"][i]), int(r["is_primary"][i]), read_names[int(r["read_id"][i])], chrom_names[int(r["chrom"][i])])
            for i in range(len(r["chrom"]))]
    return out, rows


def diff_extract(ref_cand, ref_rows, got_cand, got_rows):
    msgs = []
    for k in ("DEL", "INS", "DUP", "INV", "TRA"):
        a = collections.Counter((tuple(float(x) if isinstance(x, (int, float)) and not isinstance(x, bool) else x for x in t)) for t in ref_cand[k])
        b = collections.Counter((tuple(float(x) if isinstance(x, (int, float)) and not isinstance(x, bool) else x for x in t)) for t in got_cand[k])
        if a != b:
            msgs.append("%s: %d ref vs %d got; only-ref %s only-got %s" % (k, sum(a.values()), sum(b.values()), list((a - b).items())[:3],
                                                                          list((b - a).items())[:3]))
    if collections.Counter(ref_rows) != collections.Counter(got_rows):
        msgs.append("reads rows differ: %d vs %d" % (len(ref_rows), len(got_rows)))
    return msgs
