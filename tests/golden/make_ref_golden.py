#!/usr/bin/env python
"""Regenerates tests/golden/ref_pin.npz: the reference's own compiled hot path (oracle/_ref/libdso_ref.so, built by oracle/ref_build.sh from
the reference's sources) run through tests/test_ref_pin.py, every result it returns recorded (tests/refgold.py).  The test file runs as
usual meanwhile, so the oracle is compared with the live reference before its results are stored.

Run from the repo root, with the reference build present:  python tests/golden/make_ref_golden.py
"""
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import refgold  # noqa: E402


class _Save:
    def pytest_sessionfinish(self, session, exitstatus):
        if exitstatus != 0:
            print("make_ref_golden: the oracle disagrees with the reference; nothing stored")
            return
        refgold.save(refgold.recorded_logs(session.config))
        print(f"{refgold.GOLDEN}: {os.path.getsize(refgold.GOLDEN) / 1024:.0f} KiB")


def main():
    os.environ["DMV_REF_RECORD"] = "1"
    return pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_ref_pin.py")], plugins=[_Save()])


if __name__ == "__main__":
    sys.exit(main())
