"""CPU: the extraction logic (cutesv_b200/csrc/extract_core.h through the emulator) against golden
tuples produced by the REAL reference's parse_read."""
import functools
import gzip
import json
import os

import pytest

import emul_lib
import golden_util
from cutesv_b200 import _abi, packing, synth
from oracle import compare_extract


EXTRACT_GOLDENS = ["extract_s0", "extract_s1", "extract_s2", "extract_s3", "extract_s4", "extract_s5", "extract_s6",
                   "extract_l0", "extract_l1", "extract_l2", "extract_l3", "extract_l4"]


def _run(seed, n, p, kind="short"):
    reads, names, lens = synth.synth_alignments_long(seed, n) if kind == "long" else synth.synth_alignments(seed, n)
    rnames = sorted(set(r.query_name for r in reads))
    rid = {nm: i for i, nm in enumerate(rnames)}
    cid = {nm: i for i, nm in enumerate(names)}
    pk = packing.pack_alignments(reads, cid, rid)
    ex = emul_lib.extract(p, pk)
    cigar_of = lambda rec: (pk["cigar"][pk["cigar_off"][rec]:pk["cigar_off"][rec + 1]], int(pk["ref_start"][rec]))
    return reads, compare_extract.tuples_from_columns(ex, names, rnames, lambda rec: reads[rec].query_sequence, cigar_of,
                                                      (p.min_siglength, p.merge_ins_threshold)), ex


@pytest.mark.parametrize("name", EXTRACT_GOLDENS)
def test_emulator_matches_reference_golden(name):
    """short packets: every flag / strand branch at scale; long ones (extract_l*): BASELINE config-5-shaped records
    (>= 10^4 CIGAR ops, clips on both ends, 2-6 SA segments in every strand pattern, MaxSize -1, chains of > 64 merged
    insertions whose sequence the host rebuilds from the CIGAR)."""
    meta = json.load(open(os.path.join(golden_util.GOLDEN, name + ".json")))
    p = _abi.default_params(**meta["params"])
    reads, (gc, gr), ex = _run(meta["seed"], meta["n_reads"], p, meta.get("kind", "short"))
    if name in ("extract_l0", "extract_l1", "extract_l4"):
        assert (ex["pieces"][:, 3] == 2).any(), "the chained-insertion spill path should be exercised"
    ref_c = {k: [tuple(t) for t in v] for k, v in meta["candidate"].items()}
    ref_r = [tuple(t) for t in meta["rows"]]
    assert not compare_extract.diff_extract(ref_c, ref_r, gc, gr)


@functools.lru_cache(maxsize=None)
def _live_goldens():
    with gzip.open(os.path.join(golden_util.GOLDEN, "extract_live.json.gz"), "rt") as f:
        return json.load(f)


@pytest.mark.parametrize("seed", range(500, 520))
def test_emulator_matches_live_reference(seed):
    """A random flag setting per seed: the reference's parse_read output on the same packet, INS sequences compared by
    digest (tests/golden/extract_live.json.gz, oracle/gen_ref_golden.py)."""
    meta = _live_goldens()[str(seed)]
    p = _abi.default_params(**meta["params"])
    reads, (gc, gr), _ = _run(seed, meta["n_reads"], p)
    ref_c = {k: [tuple(t) for t in v] for k, v in meta["candidate"].items()}
    ref_r = [tuple(t) for t in meta["rows"]]
    assert not compare_extract.diff_extract(ref_c, ref_r, compare_extract.digest_ins_seqs(gc), gr)


def test_acquire_clip_pos():
    assert packing.acquire_clip_pos("10S100M5D20M3S") == (10, 3, 125)
    assert packing.acquire_clip_pos("10H100M") == (0, 0, 100)
    assert packing.acquire_clip_pos("5=2X3I4S") == (0, 4, 7)
