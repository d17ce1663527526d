"""Differential fuzzing of the HOST-SIDE logic against the live reference (authoring container only: needs
/root/reference): random shapes, ridge values, centring flags, view weights, confounds, feature groups, dtypes.
The kernels are replaced by tests/fake_ops.py (torch CPU), so every mismatch is a divergence of the Python between
the kernels from the reference's behaviour.  Ill-posed draws (c = 0 with a rank-deficient or under-determined view,
where the reference itself returns noise-dependent output) are reported only with --all.

    python tools/fuzz_vs_reference.py [seed] [trials] [--all]
"""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import fake_ops  # noqa: E402  (before refshim: the reference has its own `tests` package)
from tests import fuzz_cases as F  # noqa: E402
from oracle import refshim  # noqa: E402

refshim.install()
import cca_zoo.linear as ref  # noqa: E402

fake_ops.install(pytest.MonkeyPatch())
from cca_zoo_b200 import linear as ours  # noqa: E402


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    seed = int(args[0]) if args else 0
    trials = int(args[1]) if len(args) > 1 else 300
    show_all = "--all" in sys.argv
    medium = "--medium" in sys.argv        # wider views, explicit solver routes (top-k route needs 4k <= width)
    bad = 0
    for t in F.linear_trials(seed, trials, medium):
        msg = F.linear_mismatch(F.linear_reduce(F.linear_record(ref, t), t), F.linear_record(ours, t, ours=True), t,
                                show_all)
        if msg:
            bad += 1
            print(msg)
    print(f"seed {seed}: {trials} trials, {bad} mismatches")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
