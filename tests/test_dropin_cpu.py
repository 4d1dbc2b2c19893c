"""CPU: the drop-in resolution_* entry points (work-dir pickles -> columns -> one cluster call -> the reference's rows)
with the kernels replaced by the pipeline emulator, against the rows the REAL reference produced (tests/golden).
The -m gpu twin is tests/test_gpu_dropin.py."""
import hashlib
import json
import os

import pytest

import golden_util
from cutesv_b200 import cuteSV_resolveDUP, cuteSV_resolveINDEL, cuteSV_resolveINV, cuteSV_resolveTRA, runtime, workdir
from emul_engine import EmulEngine
from oracle import compare
from test_gpu_dropin import _tuples


@pytest.mark.parametrize("name", ["adv001", "adv034", "adv144", "cfg3_s0p004", "sweep05", "sweep11"])
def test_resolution_entry_points_cpu(tmp_path, name):
    runtime.set_engine(EmulEngine())
    try:
        case = golden_util.load_case(name)
        p = case["params"]
        path = str(tmp_path) + "/"
        idx = workdir.write_workdir(path, _tuples(case))
        action = bool(p.genotype)
        got = {}
        for chrom in idx["DEL"]:
            got[("DEL", chrom)] = cuteSV_resolveINDEL.run_del((path, chrom, "DEL", p.min_support, p.ratio_del, p.bias_del, p.min_support_allele,
                                                               "", action, p.gt_round, p.remain_reads_ratio, idx))[1]
        for chrom in idx["INS"]:
            got[("INS", chrom)] = cuteSV_resolveINDEL.run_ins((path, chrom, "INS", p.min_support, p.ratio_ins, p.bias_ins, p.min_support_allele,
                                                               "", action, p.gt_round, p.remain_reads_ratio, idx))[1]
        for chrom in idx["INV"]:
            got[("INV", chrom)] = cuteSV_resolveINV.run_inv((path, chrom, "INV", p.min_support, p.bias_inv, p.min_size, "", action, p.max_size,
                                                             p.gt_round, idx))[1]
        for chrom in idx["DUP"]:
            got[("DUP", chrom)] = cuteSV_resolveDUP.run_dup((path, chrom, p.min_support, p.bias_dup, p.min_size, "", action, p.max_size, p.gt_round,
                                                             idx))[1]
        for chrom in idx["TRA"]:
            got[("TRA", chrom)] = cuteSV_resolveTRA.run_tra((path, chrom, p.min_support, p.ratio_tra, p.bias_tra, "", False, p.gt_round, idx))[1]
        got = {k: v for k, v in got.items() if v}
        d = compare.diff_rows(case["rows"], got)
        assert not d, "\n".join(d[:4])
    finally:
        runtime.set_engine(None)


def test_dropins_batch_one_cluster_call_per_type(tmp_path):
    """The first resolution_* call of a type clusters EVERY contig of the work dir in one C-ABI call; the other contigs' calls
    slice the cache (the reference issues one call per (type, contig), cuteSV:1113-1199)."""
    from cutesv_b200 import _resolve_common
    runtime.set_engine(EmulEngine())
    try:
        _resolve_common.clear_cache()
        case = golden_util.load_case("cfg3_s0p004")
        p = case["params"]
        path = str(tmp_path) + "/"
        idx = workdir.write_workdir(path, _tuples(case))
        assert len(idx["DEL"]) > 3
        n0 = _resolve_common.N_BATCHED_CALLS
        got = {}
        for chrom in idx["DEL"]:
            got[("DEL", chrom)] = cuteSV_resolveINDEL.run_del((path, chrom, "DEL", p.min_support, p.ratio_del, p.bias_del, p.min_support_allele,
                                                               "", bool(p.genotype), p.gt_round, p.remain_reads_ratio, idx))[1]
        assert _resolve_common.N_BATCHED_CALLS - n0 == 1
        for chrom in idx["DUP"]:
            got[("DUP", chrom)] = cuteSV_resolveDUP.run_dup((path, chrom, p.min_support, p.bias_dup, p.min_size, "", bool(p.genotype), p.max_size,
                                                             p.gt_round, idx))[1]
        assert _resolve_common.N_BATCHED_CALLS - n0 == 2
        want = {k: v for k, v in case["rows"].items() if k[0] in ("DEL", "DUP")}
        d = compare.diff_rows(want, {k: v for k, v in got.items() if v})
        assert not d, "\n".join(d[:4])
        # other parameters -> another batch
        cuteSV_resolveINDEL.run_del((path, next(iter(idx["DEL"])), "DEL", p.min_support + 1, p.ratio_del, p.bias_del, p.min_support_allele,
                                     "", bool(p.genotype), p.gt_round, p.remain_reads_ratio, idx))
        assert _resolve_common.N_BATCHED_CALLS - n0 == 3
    finally:
        runtime.set_engine(None)
        _resolve_common.clear_cache()


@pytest.mark.parametrize("name", ["cfg2_s0p002", "adv034"])
def test_reference_reads_a_repo_written_work_dir(tmp_path, name):
    """--retain_work_dir compatibility the other way round: <TYPE>.pickle + sigindex written by cutesv_b200.workdir are
    byte for byte the work dir the REAL reference's own rebuild writes from the same signatures (tests/golden/ref_workdir.json,
    oracle/gen_ref_golden.py), from which the reference produced the golden rows; so its run_del / run_ins / run_inv /
    run_dup read the same lists at the same offsets."""
    want = json.load(open(os.path.join(golden_util.GOLDEN, "ref_workdir.json")))[name]
    case = golden_util.load_case(name)
    path = str(tmp_path) + "/"
    idx = workdir.write_workdir(path, _tuples(case))
    assert json.loads(json.dumps(idx)) == want["sigs_index"]
    assert sum(idx["reads_count"].values()) > 0 and any(idx[t] for t in ("DEL", "INS", "INV", "DUP"))
    for t, digest in want["sha256"].items():
        with open("%s%s.pickle" % (path, t), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, t
