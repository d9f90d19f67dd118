"""The reference's own, unmodified unittest files run against the drop-in package (tools/run_reference_tests.py).

Those files belong to the reference project, not to this repository: the test runs when LOCOHD_REFERENCE_TESTS names
the tests/ directory of a reference checkout and skips otherwise.  The known answers they check are restated, with the
repository, in test_api_dropin.py (drop-in API) and test_oracle_kat.py (oracle).  The runner was run once on a B200
with the three files: 13 passed, 1 skipped upstream (profiles/r8b_reference_tests.json, checksums of the files in
profiles/r8b_reference_tests.sha256)."""
import importlib.util
import os
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
REF_TESTS = os.environ.get("LOCOHD_REFERENCE_TESTS")


@pytest.mark.skipif(not REF_TESTS, reason="LOCOHD_REFERENCE_TESTS (tests/ of a reference checkout) is not set")
def test_reference_unittests_against_the_dropin():
    spec = importlib.util.spec_from_file_location("_run_reference_tests", ROOT / "tools" / "run_reference_tests.py")
    runner = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(runner)
    out = runner.run(Path(REF_TESTS))
    assert out["run"] == 14 and out["skipped"] == ["TestLoCoHDValues.test_consistency"]
    if out["cuda_devices"] > 0:
        assert out["not_passed"] == [] and out["passed"] == 13
    else:
        # host-side classes pass without a device; the two scoring tests fail loudly - there is no CPU fallback
        assert out["passed"] == 11
        assert sorted(t for t, _ in out["not_passed"]) == ["TestLoCoHDValues.test_small_locohd", "TestTagPairingRule.test_in_locohd"]
        assert all("no CPU fallback" in msg for _, msg in out["not_passed"])
