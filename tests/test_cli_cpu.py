"""CPU: CLI flag surface identical to the reference's parseArgs; task windows like cuteSV:1018-1044."""
import json
import os

import golden_util
from cutesv_b200 import cli


def test_defaults_and_flags_match_reference():
    """The namespace the reference's parseArgs returned for the same argument lists (tests/golden/ref_cli_args.json,
    oracle/gen_ref_golden.py)."""
    cases = json.load(open(os.path.join(golden_util.GOLDEN, "ref_cli_args.json")))
    assert len(cases) == 2
    for case in cases:
        got = vars(cli.build_parser().parse_args(case["argv"]))
        assert got == case["args"]
        assert {k: type(v) for k, v in got.items()} == {k: type(v) for k, v in case["args"].items()}


def test_task_windows_float_bounds():
    stats = [("c1", 1000, 0, 1000), ("c2", 1, 0, 1)]
    lens = {"c1": 25000000, "c2": 5000}
    tasks, info = cli.task_windows(stats, lambda n: lens[n], 16, 10000000)
    assert info == [["c1", 25000000], ["c2", 5000]]
    assert tasks[-1] == ["c2", 0, 5000]
    c1 = [t for t in tasks if t[0] == "c1"]
    unit = 1001 / 16 / 10
    batch = 25000000 / (int(1000 / unit) + 1)   # coverage-balanced float window size, cuteSV:1034
    assert c1[0][1] == 0 and c1[0][2] == batch
    for x, y in zip(c1, c1[1:]):
        assert y[1] == x[2]                        # contiguous, float bounds preserved
    assert c1[-1][2] in (25000000, c1[-1][1] + batch)


def test_params_from_args():
    a = cli.build_parser().parse_args(["a", "b", "c", "d", "-s", "3", "--genotype"])
    p = cli.params_from_args(a)
    assert p.min_support == 3 and p.min_support_allele == 3 and p.genotype == 1 and p.bias_del == 200
