"""Goldens for the tests that used to call the reference directly: its command-line parser, its VCF header, the work
dir its own rebuild writes, and its parse_read on seeded short-read packets.  Only the reference's OUTPUT is committed
(INS sequences as SHA-256 prefixes); the inputs are regenerated from the seeds and argument lists stored beside it.
Needs the reference sources (see ref_harness.py):  python -m oracle.gen_ref_golden"""
import gzip
import hashlib
import io
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cutesv_b200 import _abi, synth  # noqa: E402
from oracle import compare_extract, ref_harness  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

CLI_ARGVS = [
    ["a.bam", "r.fa", "o.vcf", "wd"],
    ["a.bam", "r.fa", "o.vcf", "wd", "--genotype", "-s", "3", "-l", "50", "-L", "-1", "-t", "4", "-b", "500", "-p", "-1", "-q", "10",
     "-r", "100", "-md", "500", "-mi", "500", "-sl", "20", "--max_cluster_bias_INS", "1000", "--diff_ratio_merging_INS", "0.9",
     "--max_cluster_bias_DEL", "1000", "--diff_ratio_merging_DEL", "0.5", "--max_cluster_bias_INV", "7", "--max_cluster_bias_DUP", "8",
     "--max_cluster_bias_TRA", "9", "--diff_ratio_filtering_TRA", "0.5", "--remain_reads_ratio", "0.7", "--report_readid",
     "--ignore_sequence", "--retain_work_dir", "--write_old_sigs", "-S", "HG002", "--gt_round", "100", "-include_bed", "x.bed"],
]
VCF_HEADER = dict(contigs=[["1", 1000], ["X", 77]], sample="NULL", argv=["a.bam", "r.fa", "o.vcf", "w", "--genotype"])
WORKDIR_CASES = ["cfg2_s0p002", "adv034"]
LIVE_EXTRACT_SEEDS = range(500, 520)
LIVE_EXTRACT_READS = 120


def live_extract_params(seed):
    """A random flag setting per seed (the extraction flags of parseArgs)."""
    rng = np.random.default_rng(seed)
    return dict(min_size=int(rng.choice([30, 50, 10])), max_size=int(rng.choice([-1, 100000, 2000])),
                min_mapq=int(rng.choice([20, 0, 30])), max_split_parts=int(rng.choice([7, -1, 2, 3])),
                min_read_len=int(rng.choice([500, 100])), min_siglength=int(rng.choice([10, 30])),
                merge_del_threshold=int(rng.choice([0, 500])), merge_ins_threshold=int(rng.choice([100, 500, 0])))


def sha256_file(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def main():
    import golden_util
    ref_harness.modules()   # also puts the reference's package on sys.path
    from cuteSV.cuteSV_Description import Generation_VCF_header, parseArgs

    cli = [dict(argv=argv, args=vars(parseArgs(argv))) for argv in CLI_ARGVS]
    with open(os.path.join(OUT, "ref_cli_args.json"), "w") as f:
        json.dump(cli, f, indent=1)

    buf = io.StringIO()
    Generation_VCF_header(buf, VCF_HEADER["contigs"], VCF_HEADER["sample"], VCF_HEADER["argv"])
    with open(os.path.join(OUT, "ref_vcf_header.json"), "w") as f:
        json.dump(dict(VCF_HEADER, lines=buf.getvalue().splitlines()), f, indent=1)

    # the work dir the reference's own rebuild writes from a golden case's inputs: its index and the bytes of every file
    wd = {}
    for name in WORKDIR_CASES:
        case = golden_util.load_case(name)
        tuples = ref_harness.to_tuples(case["sigs"], case["reads"], case["names"], synth.read_name)
        with tempfile.TemporaryDirectory() as d:
            idx = ref_harness.write_reference_workdir(d + "/", tuples)
            files = {t: sha256_file("%s/%s.pickle" % (d, t)) for t in ("DEL", "INS", "DUP", "INV", "TRA", "reads")}
        wd[name] = dict(sigs_index=idx, sha256=files)
    with open(os.path.join(OUT, "ref_workdir.json"), "w") as f:
        json.dump(wd, f, indent=1)

    live = {}
    for seed in LIVE_EXTRACT_SEEDS:
        kw = live_extract_params(seed)
        reads, _, _ = synth.synth_alignments(seed, LIVE_EXTRACT_READS)
        c, r = ref_harness.run_parse_reads(reads, _abi.default_params(**kw))
        c = compare_extract.digest_ins_seqs(c)
        live[str(seed)] = dict(n_reads=LIVE_EXTRACT_READS, params=kw, candidate={k: [list(t) for t in v] for k, v in c.items()},
                               rows=[list(t) for t in r])
    with gzip.GzipFile(os.path.join(OUT, "extract_live.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(live, sort_keys=True).encode())
    print("cli", len(cli), "workdir", sorted(wd), "live extract seeds", len(live))


if __name__ == "__main__":
    main()
