"""Runs the UNMODIFIED reference (/root/reference/src) on columnar inputs (TEST INFRASTRUCTURE).

Only usable where the reference sources are present, so this module is imported by the golden
generators (oracle/gen_*.py), which commit the reference's outputs under tests/golden/; the tests
compare against those files and never import the reference.

pysam / cigar / Bio are not installed here; they are stubbed with the minimal surface the hot
path touches (SURVEY.md section 8c).
"""
import importlib.machinery
import importlib.util
import os
import pickle
import re
import sys
import tempfile
import types

REF_SRC = "/root/reference/src"


def available():
    return os.path.isdir(os.path.join(REF_SRC, "cuteSV"))


def _install_stubs():
    if "pysam" not in sys.modules:
        # the test-only fake pysam (constants + pickle-backed AlignmentFile / FastaFile)
        fake = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "fake_pysam", "pysam.py")
        spec = importlib.util.spec_from_file_location("pysam", fake)
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        sys.modules["pysam"] = m
    if "cigar" not in sys.modules:
        m = types.ModuleType("cigar")

        class Cigar(object):  # PyPI "Cigar": Cigar(s).items() -> (length, op) pairs
            def __init__(self, s):
                self.s = s

            def items(self):
                for n, op in re.findall(r"(\d+)([MIDNSHP=X])", self.s):
                    yield (int(n), op)
        m.Cigar = Cigar
        sys.modules["cigar"] = m
    if "Bio" not in sys.modules:
        bio = types.ModuleType("Bio")
        seqm = types.ModuleType("Bio.Seq")
        comp = str.maketrans("ACGTNacgtn", "TGCANtgcan")

        class Seq(object):
            def __init__(self, s):
                self.s = s

            def reverse_complement(self):
                return Seq(self.s.translate(comp)[::-1])

            def __str__(self):
                return self.s
        seqm.Seq = Seq
        bio.Seq = seqm
        sys.modules["Bio"] = bio
        sys.modules["Bio.Seq"] = seqm


_mods = {}


def modules():
    """(main_script_module, resolveINDEL, resolveDUP, resolveINV, resolveTRA, genotype)."""
    if not _mods:
        if not available():
            raise RuntimeError("reference not present at %s" % REF_SRC)
        _install_stubs()
        if REF_SRC not in sys.path:
            sys.path.insert(0, REF_SRC)
        from cuteSV import cuteSV_genotype, cuteSV_resolveDUP, cuteSV_resolveINDEL, cuteSV_resolveINV, cuteSV_resolveTRA
        loader = importlib.machinery.SourceFileLoader("cutesv_ref_main", os.path.join(REF_SRC, "cuteSV", "cuteSV"))
        spec = importlib.util.spec_from_loader("cutesv_ref_main", loader)
        main = importlib.util.module_from_spec(spec)
        sys.modules["cutesv_ref_main"] = main  # multiprocessing pickles its functions by module name
        loader.exec_module(main)
        _mods.update(main=main, indel=cuteSV_resolveINDEL, dup=cuteSV_resolveDUP, inv=cuteSV_resolveINV,
                     tra=cuteSV_resolveTRA, genotype=cuteSV_genotype)
    return _mods


def ins_seq_of(key, n):
    """Deterministic synthetic INS sequence of length n.  `key` must be a function of the
    signature's content (see ins_key) so that identical tuples carry identical sequences."""
    pat = "ACGT"
    k = key % 4
    s = (pat[k:] + pat[:k]) * (n // 4 + 1)
    return s[:n]


def ins_key(ins_cols, i):
    return int(ins_cols["a"][i]) + int(ins_cols["read_id"][i]) + int(ins_cols["b"][i])


def ins_seq_fn(ins_cols):
    """idx -> synthetic sequence of INS signature idx (what a host packer would hold)."""
    return lambda i: ins_seq_of(ins_key(ins_cols, i), int(ins_cols["c"][i]))


def to_tuples(sigs, reads, chrom_names, read_name):
    """Columnar arrays -> the reference's tuple lists (cuteSV:520-531,235-239,55-60,111-117,733)."""
    out = {k: [] for k in ("DEL", "INS", "DUP", "INV", "TRA")}
    s = sigs.get("DEL")
    if s is not None:
        for i in range(len(s["chrom"])):
            out["DEL"].append((int(s["a"][i]), int(s["b"][i]), read_name(int(s["read_id"][i])), "DEL",
                               chrom_names[int(s["chrom"][i])]))
    s = sigs.get("INS")
    if s is not None:
        for i in range(len(s["chrom"])):
            a = int(s["a"][i])
            pos = a // 2 if a % 2 == 0 else a / 2
            out["INS"].append((pos, int(s["b"][i]), read_name(int(s["read_id"][i])), ins_seq_of(ins_key(s, i), int(s["c"][i])),
                               "INS", chrom_names[int(s["chrom"][i])]))
    s = sigs.get("DUP")
    if s is not None:
        for i in range(len(s["chrom"])):
            out["DUP"].append((int(s["a"][i]), int(s["b"][i]), read_name(int(s["read_id"][i])), "DUP",
                               chrom_names[int(s["chrom"][i])]))
    s = sigs.get("INV")
    if s is not None:
        for i in range(len(s["chrom"])):
            out["INV"].append(("++" if int(s["c"][i]) == 0 else "--", int(s["a"][i]), int(s["b"][i]),
                               read_name(int(s["read_id"][i])), "INV", chrom_names[int(s["chrom"][i])]))
    s = sigs.get("TRA")
    if s is not None:
        for i in range(len(s["chrom"])):
            c = int(s["c"][i])
            out["TRA"].append(("ABCD"[c & 3], int(s["a"][i]), chrom_names[c >> 2], int(s["b"][i]),
                               read_name(int(s["read_id"][i])), "TRA", chrom_names[int(s["chrom"][i])]))
    rl = []
    if reads is not None:
        for i in range(len(reads["chrom"])):
            rl.append((int(reads["start"][i]), int(reads["end"][i]), int(reads["is_primary"][i]),
                       read_name(int(reads["read_id"][i])), chrom_names[int(reads["chrom"][i])]))
    out["reads"] = rl
    return out


def sorted_alignments(reads):
    """The reads table as an all-alignments table in BAM order (contig id, start; stable)."""
    import numpy as np
    order = np.lexsort((np.arange(len(reads["chrom"])), reads["start"], reads["chrom"]))
    return {k: v[order] for k, v in reads.items()}


def write_fake_bam(path, aln, chrom_names, lens, read_name):
    """aln: all-alignments table (BAM order) -> pickle readable by tests/fake_pysam (TRA genotyper input)."""
    from cutesv_b200.synth import SynthRead
    recs = []
    for i in range(len(aln["chrom"])):
        r = SynthRead()
        r.reference_name = chrom_names[int(aln["chrom"][i])]
        r.reference_start = int(aln["start"][i])
        r.reference_end = int(aln["end"][i])
        r.flag = 0 if int(aln["is_primary"][i]) else 2048
        r.query_name = read_name(int(aln["read_id"][i]))
        r.mapq, r.query_length, r.query_sequence, r.cigartuples, r.cigar, r.tags = 60, 0, "", [], [], []
        recs.append(r)
    with open(path, "wb") as f:
        pickle.dump(dict(contigs=[(n, int(l)) for n, l in zip(chrom_names, lens)], reads=recs), f)


def write_reference_workdir(tmp, tuples, n_pids=1):
    """The reference's work dir under `tmp` (ends in "/"): per-worker signature pickles, then its rebuild
    (process_process_sigs_type, cuteSV:750-857) into <TYPE>.pickle.  Returns sigs_index."""
    main = modules()["main"]
    os.mkdir(tmp + "signatures")
    pids = list(range(100, 100 + n_pids))
    for k in ("DEL", "INS", "DUP", "INV", "TRA", "reads"):
        lst = tuples[k]
        for j, pid in enumerate(pids):  # round-robin "tasks" over fake worker pids
            with open("%ssignatures/%s%s.pickle" % (tmp, pid, k), "ab") as f:
                pickle.dump(lst[j::n_pids], f)
    sigs_index = {}
    for k in ("DEL", "INS", "DUP", "INV", "TRA", "reads"):
        r = main.process_process_sigs_type((k, tmp, pids, False))
        sigs_index[r[0]] = r[1]
        if r[0] == "reads":
            sigs_index["reads_count"] = r[2]
    return sigs_index


def run_reference(sigs, reads, chrom_names, read_name, p, types_=("DEL", "INS", "INV", "DUP", "TRA"),
                  n_pids=1, tra_bam=None):
    """Reference rebuild (process_process_sigs_type, cuteSV:750-857) + clustering phase
    (cuteSV:1113-1199, run serially).  p: csv_params.  Returns {(type, chrom): rows}.

    TRA is run with action=False unless tra_bam (a fake-pysam BAM path) is given: its call_gt
    re-opens the BAM."""
    m = modules()
    tuples = to_tuples(sigs, reads, chrom_names, read_name)
    res = {}
    with tempfile.TemporaryDirectory() as d:
        tmp = d + "/"
        sigs_index = write_reference_workdir(tmp, tuples, n_pids)
        action = bool(p.genotype)
        if "DEL" in types_:
            for chr_ in sigs_index["DEL"]:
                c, rows = m["indel"].run_del((tmp, chr_, "DEL", p.min_support, p.ratio_del, p.bias_del,
                                              p.min_support_allele, "", action, p.gt_round, p.remain_reads_ratio,
                                              sigs_index))
                res[("DEL", c)] = rows
        if "INS" in types_:
            for chr_ in sigs_index["INS"]:
                c, rows = m["indel"].run_ins((tmp, chr_, "INS", p.min_support, p.ratio_ins, p.bias_ins,
                                              p.min_support_allele, "", action, p.gt_round, p.remain_reads_ratio,
                                              sigs_index))
                res[("INS", c)] = rows
        if "INV" in types_:
            for chr_ in sigs_index["INV"]:
                c, rows = m["inv"].run_inv((tmp, chr_, "INV", p.min_support, p.bias_inv, p.min_size, "", action,
                                            p.max_size, p.gt_round, sigs_index))
                res[("INV", c)] = rows
        if "DUP" in types_:
            for chr_ in sigs_index["DUP"]:
                c, rows = m["dup"].run_dup((tmp, chr_, p.min_support, p.bias_dup, p.min_size, "", action,
                                            p.max_size, p.gt_round, sigs_index))
                res[("DUP", c)] = rows
        if "TRA" in types_:
            for chr_ in sigs_index["TRA"]:
                c, rows = m["tra"].run_tra((tmp, chr_, p.min_support, p.ratio_tra, p.bias_tra, tra_bam or "",
                                            bool(tra_bam) and bool(p.genotype), p.gt_round, sigs_index))
                res[("TRA", c)] = rows
    return res


def run_parse_reads(reads, p):
    """The reference's extraction loop body (single_pipe, cuteSV:709-733) on in-memory read objects:
    calls the UNMODIFIED parse_read (cuteSV:606-681).  Returns (candidate dict, reads_info_list)."""
    main = modules()["main"]
    candidate = {k: [] for k in ("DEL", "INS", "DUP", "INV", "TRA")}
    rows = []
    for read in reads:
        if read.flag == 256 or read.flag == 272:
            continue
        main.parse_read(read, candidate, read.reference_name, p.min_size, p.min_mapq, p.max_split_parts, p.min_read_len,
                        p.min_siglength, p.merge_del_threshold, p.merge_ins_threshold, p.max_size)
        if read.mapq >= p.min_mapq:
            rows.append((read.reference_start, read.reference_end, 1 if read.flag in (0, 16) else 0, read.query_name,
                         read.reference_name))
    return candidate, rows


class _Args(object):
    pass


def reference_vcf_lines(results_by_chrom, ref_seqs, genotype, max_size=100000, min_size=30, report_readid=False, ignore_sequence=False):
    """The reference's generate_output (cuteSV_genotype.py:242-467) + the SVID loop of main_ctrl
    (cuteSV:1208-1237) on in-memory rows, with pysam.FastaFile stubbed by `ref_seqs`."""
    import copy
    m = modules()
    pys = sys.modules["pysam"]

    class FastaFile(object):
        def __init__(self, path):
            pass

        def fetch(self, chrom):
            return ref_seqs[chrom]

        def close(self):
            pass
    pys.FastaFile = FastaFile
    args = _Args()
    args.genotype, args.max_size, args.min_size = genotype, max_size, min_size
    args.report_readid, args.ignore_sequence = report_readid, ignore_sequence
    lines = []
    svid = {"INS": 0, "DEL": 0, "BND": 0, "DUP": 0, "INV": 0}
    with tempfile.TemporaryDirectory() as d:
        tmp = d + "/"
        os.mkdir(tmp + "results")
        for chrom in sorted(results_by_chrom):
            m["genotype"].generate_output(args, copy.deepcopy(results_by_chrom[chrom]), "ref.fa", chrom, tmp)
        for chrom in sorted(results_by_chrom):
            with open("%sresults/%s.pickle" % (tmp, chrom), "rb") as f:
                while True:
                    try:
                        for svtype, line in pickle.load(f):
                            lines.append(line.replace("<SVID>", str(svid[svtype])))
                            svid[svtype] += 1
                    except EOFError:
                        break
    return lines
