"""The parity sink (SURVEY appendix B): rows -> VCF records, against lines produced by the REAL
reference's generate_output + SVID loop (tests/golden/vcf_*.json).  CPU: formatter on the golden
rows; GPU: rows computed by the CUDA path -> bit-identical VCF body."""
import json
import os

import pytest

import golden_util
import vcf_util
from cutesv_b200 import vcf

CASES = ["adv034", "adv144", "cfg3_s0p004", "cfg2_s0p002"]


def _golden_lines(name):
    return json.load(open(os.path.join(golden_util.GOLDEN, "vcf_%s.json" % name)))


def _lines(case, rows):
    byc = vcf_util.rows_by_chrom(rows)
    refseq = vcf_util.synthetic_reference(case["names"], [min(int(x), 6000000) for x in case["lens"]])
    opts = dict(genotype=bool(case["params"].genotype), max_size=100000, min_size=30, report_readid=False, ignore_sequence=False)
    return vcf.assign_ids({c: vcf.format_records(r, refseq[c], opts) for c, r in byc.items()})


@pytest.mark.parametrize("name", CASES)
def test_formatter_matches_reference_lines(name):
    case = golden_util.load_case(name)
    assert _lines(case, case["rows"]) == _golden_lines(name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_cuda_rows_give_identical_vcf(engine, name):
    case = golden_util.load_case(name)
    engine.set_params(case["params"])
    engine.set_contigs(case["lens"])
    res = engine.cluster(case["sigs"], case["reads"])
    got = golden_util.to_rows(case, res)
    a, b = _lines(case, got), _golden_lines(name)
    # DUP/BND RNAMES are not printed by default, so the record text must be identical
    assert a == b


def test_header_shape():
    h = vcf.header_lines([("1", 100), ("2", 50)], "S1", ["in.bam", "ref.fa", "out.vcf", "wd"], date="D")
    assert h[0] == "##fileformat=VCFv4.2" and h[2] == "##fileDate=D"
    assert h[3] == "##contig=<ID=1,length=100>"
    assert h[-1].endswith("FORMAT\tS1") and h[-2] == '##CommandLine="cuteSV in.bam ref.fa out.vcf wd"'
    assert sum(1 for x in h if x.startswith("##INFO")) == 12 and sum(1 for x in h if x.startswith("##FORMAT")) == 5


def test_header_matches_reference_when_present():
    """Header lines the reference's Generation_VCF_header wrote (tests/golden/ref_vcf_header.json, oracle/gen_ref_golden.py)."""
    case = json.load(open(os.path.join(golden_util.GOLDEN, "ref_vcf_header.json")))
    ref = case["lines"]
    got = vcf.header_lines(case["contigs"], case["sample"], case["argv"])[:-1]
    assert len(ref) == len(got)
    for a, b in zip(ref, got):
        if a.startswith("##fileDate"):
            continue
        assert a == b


def test_indexed_fasta_equals_full_load(tmp_path):
    """vcf.IndexedFasta (random access, .fai or on-the-fly index) vs read_fasta on every access pattern format_records uses."""
    import numpy as np
    from cutesv_b200 import vcf
    rng = np.random.default_rng(3)
    seqs = {"chrA": "".join(rng.choice(list("ACGTN"), 1234)), "chrB": "".join(rng.choice(list("acgtRY"), 60)), "c3": "A", "chrD": "".join(rng.choice(list("ACGT"), 601))}
    fa = tmp_path / "r.fa"
    with open(fa, "w") as f:
        for k, v in seqs.items():
            f.write(">%s some description\n" % k)
            for i in range(0, len(v), 60):
                f.write(v[i:i + 60] + "\n")
    full = vcf.read_fasta(str(fa))
    assert full == seqs
    for use_fai in (False, True):
        if use_fai:   # a samtools-style index
            off = 0
            lines = []
            data = open(fa, "rb").read()
            for k, v in seqs.items():
                off = data.index((">%s some description\n" % k).encode()) + len(">%s some description\n" % k)
                lines.append("%s\t%d\t%d\t%d\t%d\n" % (k, len(v), off, min(60, len(v)), min(60, len(v)) + 1))
            open(str(fa) + ".fai", "w").write("".join(lines))
        idx = vcf.IndexedFasta(str(fa))
        assert "chrA" in idx and "nope" not in idx
        for k, v in seqs.items():
            s = idx[k]
            assert len(s) == len(v)
            for _ in range(200):
                a, b = sorted(int(x) for x in rng.integers(0, len(v) + 5, 2))
                assert s[a:b] == v[a:b], (k, a, b)
                i = int(rng.integers(0, len(v)))
                assert s[i] == v[i]
            assert s[5:2] == "" and s[len(v):len(v) + 3] == ""
            with pytest.raises(IndexError):
                s[len(v)]
        idx.close()
    ragged = tmp_path / "ragged.fa"
    ragged.write_text(">x\nACGT\nAC\nACGTAC\n>y\nTT\n")
    idx = vcf.IndexedFasta(str(ragged))   # not indexable: falls back to the full load
    assert idx["x"] == "ACGTACACGTAC" and idx["y"][0:2] == "TT"
    idx.close()
