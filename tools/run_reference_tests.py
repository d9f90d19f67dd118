"""Runs the reference's OWN, unmodified unittest files (tests/test_wfs.py, test_tag_pairing_rule.py, test_locohd.py of
fazekaszs/loco_hd) against this repository's drop-in `loco_hd` package.

    python tools/run_reference_tests.py [DIR]      DIR: tests/ of a reference checkout ($LOCOHD_REFERENCE_TESTS)

The files are loaded by path (so that `import loco_hd` inside them resolves to this repository, not to the reference's
pure-Python package directory next to them); nothing is copied.  Prints one JSON line: tests run, passed, skipped, and
for every error / failure the test id and the first line of the message.  On a box without a CUDA device the two tests
that score (test_small_locohd, test_in_locohd) must fail with the library's loud "no CPU fallback" RuntimeError - the
host-side classes (weight functions, tag pairing rules, constructor validation) need no device.
`test_consistency` is skipped upstream unless requested (its golden outputs are missing from the reference checkout).
"""
import importlib.util
import io
import json
import os
import sys
import unittest
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
FILES = ("test_wfs", "test_tag_pairing_rule", "test_locohd")


def run(test_dir: Path) -> dict:
    if str(ROOT) not in sys.path:
        sys.path.insert(0, str(ROOT))
    import loco_hd

    assert Path(loco_hd.__file__).resolve().parent == ROOT / "loco_hd", "the drop-in package must be the one under test"
    suite = unittest.TestSuite()
    for name in FILES:
        spec = importlib.util.spec_from_file_location("reference_" + name, test_dir / f"{name}.py")
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        suite.addTests(unittest.defaultTestLoader.loadTestsFromModule(mod))
    res = unittest.TextTestRunner(stream=io.StringIO(), verbosity=0).run(suite)
    bad = [(t.id().split(".", 1)[1], msg.strip().splitlines()[-1]) for t, msg in res.errors + res.failures]
    return {"dir": str(test_dir), "run": res.testsRun, "passed": res.testsRun - len(bad) - len(res.skipped),
            "skipped": [t.id().split(".", 1)[1] for t, _ in res.skipped], "not_passed": bad,
            "cuda_devices": loco_hd.loco_hd.device_count()}


if __name__ == "__main__":
    d = Path(sys.argv[1] if len(sys.argv) > 1 else os.environ["LOCOHD_REFERENCE_TESTS"])
    out = run(d)
    print(json.dumps(out))
    sys.exit(0 if not out["not_passed"] else 1)
