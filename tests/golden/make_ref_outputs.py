"""Regenerates tests/golden/ref_outputs.npz, the reference's outputs that tests/test_oracle_vs_ref.py and the reference
checks of tests/test_host_logic.py compare with.  Needs the reference library built from an ImageMagick 7.1.1-45 source
tree (oracle/_ref/libmagickref.so) and the product library (`IMAGEMAGICK_SOURCE=<tree> python __graft_entry__.py`).
Runs those tests against the live library (MB200_RECORD_REF_OUTPUTS=1); the file is rewritten only when every one of
them ran and passed.

    python tests/golden/make_ref_outputs.py
"""
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
TESTS = ["tests/test_oracle_vs_ref.py",
         "tests/test_host_logic.py::test_sharpen_and_edge_kernels_match_the_reference_taps",
         "tests/test_host_logic.py::test_motion_blur_taps_and_offsets_match_the_reference"]


class Outcomes:
    def __init__(self):
        self.ran, self.not_passed = 0, []

    def pytest_runtest_logreport(self, report):
        if report.when == "call" and report.passed:
            self.ran += 1
        elif report.skipped or report.failed:
            self.not_passed.append(f"{report.nodeid}: {report.outcome}")


if __name__ == "__main__":
    for lib in ("oracle/_ref/libmagickref.so", "imagemagick_b200/lib/libmagickb200.so"):
        if not (ROOT / lib).exists():
            sys.exit(f"{lib} is not built")
    os.environ["MB200_RECORD_REF_OUTPUTS"] = "1"
    os.chdir(ROOT)
    import pytest
    outcomes = Outcomes()
    rc = pytest.main(["-q", "-p", "no:cacheprovider", *TESTS], plugins=[outcomes])
    if rc != 0 or outcomes.not_passed or not outcomes.ran:
        sys.exit("not rewritten: every test must run and pass\n" + "\n".join(outcomes.not_passed))
    import util
    util.save_recording()
    print(f"{util.REF_GOLDEN.relative_to(ROOT)}: {len(util._store)} entries from {outcomes.ran} tests")
