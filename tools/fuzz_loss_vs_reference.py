"""Differential fuzzing of the objectives' HOST-SIDE logic (route selection, analytic backward) against the live
reference's forward + autograd (authoring container only).  Kernels replaced by tests/fake_ops.py.  Batches with
n - 1 <= 1.25 width (rank-deficient or barely determined batch covariance) are skipped unless --all: there the reference differentiates
through an eigendecomposition with repeated eigenvalues and its own gradient is rounding noise.

    python tools/fuzz_loss_vs_reference.py [seed] [trials] [--all]
"""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import fake_ops  # noqa: E402
from tests import fuzz_cases as F  # noqa: E402
from oracle import refshim  # noqa: E402

refshim.install()
from cca_zoo.deep import objectives as ref  # noqa: E402

fake_ops.install(pytest.MonkeyPatch())
from cca_zoo_b200.deep import objectives as ours  # noqa: E402


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    seed = int(args[0]) if args else 0
    trials = int(args[1]) if len(args) > 1 else 200
    show_all = "--all" in sys.argv
    bad = 0
    for i, t in enumerate(F.loss_trials(seed, trials)):
        if not t["determined"] and not show_all:
            continue
        msg = F.loss_mismatch(F.loss_record(ref, t, i), F.loss_record(ours, t, i), t)
        if msg:
            bad += 1
            print(msg)
    print(f"seed {seed}: {trials} trials, {bad} mismatches")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
