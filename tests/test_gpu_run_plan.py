"""The launch planner chooses what it chose when tests/golden/run_plan.json was recorded: for every handle of a grid that
crosses each of its thresholds on both sides, the same run kernel (kernel_name), block size of the CTA helper kernels
(block_threads) and pair precision, or the same create error.  The rules depend on the SM count: the file was recorded
on a B200 (148 SMs) by tests/golden/make_run_plan.py, which this test replays."""
import importlib.util
import json
import os

import pytest

from conftest import GOLDEN


def _recorder():
    spec = importlib.util.spec_from_file_location("make_run_plan", os.path.join(GOLDEN, "make_run_plan.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


pytestmark = pytest.mark.gpu


def test_run_plan_matches_recorded_choices(pm):
    with open(os.path.join(GOLDEN, "run_plan.json")) as f:
        entries = json.load(f)
    rec = _recorder()
    grid = list(rec.grid())
    assert [[e["case"], e["hint"], e["create_env"]] for e in entries] == \
        [json.loads(json.dumps(list(g[:3]))) for g in grid], "run_plan.json was recorded from another grid"
    mismatches = []
    for e, (case_kw, hint, create_env, queries) in zip(entries, grid):
        seen = rec.observe(pm, case_kw, hint, create_env, queries)
        if seen != e["seen"]:
            mismatches.append((e["case"], e["hint"], e["create_env"], e["seen"], seen))
    assert not mismatches, f"{len(mismatches)} of {len(entries)} handles differ, first: {mismatches[:3]}"
