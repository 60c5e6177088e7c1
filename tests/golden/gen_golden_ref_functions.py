#!/usr/bin/env python3
"""Writes tests/golden/ref_functions.npz: per case of tests/test_oracle_vs_ref.py, the 64-bit digests of the answers to its
seeded inputs, in the order the test produces them.  The test compares the oracle's answers with these where the reference's
compiled functions (oracle/_ref/libhmref.so) are not built.

The digests are taken from the oracle's answers while every case runs exactly as in the test, so where libhmref.so is built
each answer is first asserted equal to the reference's and the file records the reference's answers.  The committed file was
recorded without libhmref.so, from oracle sources unchanged since the commit at which the whole CPU suite - all 47 cases of
tests/test_oracle_vs_ref.py against libhmref.so among them - last passed (fbd51ed); on these inputs the oracle's answers are
therefore the reference's.  Usage: python tests/golden/gen_golden_ref_functions.py"""
import itertools
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

import _util  # noqa: E402
import test_oracle_vs_ref as t  # noqa: E402


def cases(fn):
    """the keyword arguments of every parameter set of a pytest.mark.parametrize'd test function"""
    axes = []
    for m in getattr(fn, "pytestmark", []):
        if m.name == "parametrize":
            names = [s.strip() for s in m.args[0].split(",")]
            axes.append([dict(zip(names, v if len(names) > 1 else (v,))) for v in m.args[1]])
    for combo in itertools.product(*axes):
        yield {k: v for d in combo for k, v in d.items()}


def main():
    oracle, hmref = _util.load_oracle(), _util.load_hmref()
    if hmref is None:
        print("oracle/_ref/libhmref.so is not built: recording the oracle's answers unchecked", file=sys.stderr)
    t.RECORD = {}
    for name in sorted(n for n in dir(t) if n.startswith("test_")):
        for kw in cases(getattr(t, name)):
            getattr(t, name)(oracle=oracle, hmref=hmref, **kw)
    np.savez_compressed(os.path.join(HERE, "ref_functions.npz"), **t.RECORD)
    print(f"{len(t.RECORD)} cases, {sum(len(v) for v in t.RECORD.values())} answers")


if __name__ == "__main__":
    main()
