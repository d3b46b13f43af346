"""The reference's own evidence, kept in the repository.  tests/golden/reference_tests_run_*.json record runs of the reference's OWN test
files against the executor restatement and the drop-ins (tools/run_reference_tests.py; the scenarios are carried by
tests/test_executor_reference_cases.py).  tests/golden/fuzz_*.json.gz record the reference's outputs on each differential fuzzer's seeded
inputs (`tools/<fuzzer> --record`); the fuzzers compare this repository's kernels' source (host build / warp emulator), drop-ins and batched
chain (CPU simulator) against those recordings."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_run_records_have_no_unexplained_failure():
    for name in ("framework", "dropin"):
        with open(os.path.join(ROOT, "tests", "golden", f"reference_tests_run_{name}.json")) as f:
            s = json.load(f)
        assert s["passed"] > 0 and all(v["bucket"] != "other" for v in s["not_passed_detail"].values())


@pytest.mark.parametrize("tool,recording", [("fuzz_vs_reference.py", "fuzz_toon.json.gz"), ("fuzz_mask_vs_reference.py", "fuzz_mask.json.gz"),
                                            ("fuzz_json_repair_vs_reference.py", "fuzz_json_repair.json.gz"), ("fuzz_plugins_vs_reference.py", "fuzz_plugins.json.gz"),
                                            ("fuzz_chain_vs_reference.py", "fuzz_chain.json.gz")])
def test_differential_fuzz_against_recorded_reference_outputs(tool, recording):
    """A short run of each differential fuzzer against the reference's recorded outputs on the same seeded inputs; the long live runs
    are recorded in DESIGN.md §5."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool), "--replay", os.path.join(ROOT, "tests", "golden", recording)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and " bad=0" in p.stdout, (p.stdout[-2000:], p.stderr[-2000:])
