"""Differential fuzz of the host logic against the reference's outputs, kernels replaced by tests/fake_ops.py.
A fixed seed of tests/fuzz_cases.py (the trials of tools/fuzz_vs_reference.py and tools/fuzz_loss_vs_reference.py):
random shapes, ridge values, centring flags, view weights, confounds, feature groups and dtypes must give the
reference's scores, weights, means and pairwise correlations wherever the problem is well posed and the component is
determined, and the reference's objective values and gradients wherever the batch covariance is determined.  The
reference's records are stored in tests/golden/reference_live.* (oracle/make_golden_live.py)."""
import pytest

from tests import fake_ops
from tests import fuzz_cases as F
from tests import golden_io as G

SEED, TRIALS = G.META_LIVE["fuzz_seed"], G.META_LIVE["fuzz_trials"]


@pytest.fixture
def host(monkeypatch):
    fake_ops.install(monkeypatch)


def test_fixed_seed_fuzz_has_no_mismatch(host):
    from cca_zoo_b200 import linear as ours

    trials = F.linear_trials(SEED, TRIALS)
    assert len(trials) == len(G.META_LIVE["fuzz"]) == 200
    bad = []
    for i, (t, meta) in enumerate(zip(trials, G.META_LIVE["fuzz"])):
        r = dict(meta)
        if "dtypes" in meta:
            r.update(weights=G.live_list(f"fuzz/{i}/w"), means=G.live_list(f"fuzz/{i}/mean"),
                     score=G.live(f"fuzz/{i}/score"), pairwise=G.live(f"fuzz/{i}/pairwise"))
        msg = F.linear_mismatch(r, F.linear_record(ours, t, ours=True), t)
        if msg:
            bad.append(msg)
    assert not bad, "\n".join(bad)


def test_fixed_seed_loss_fuzz_has_no_mismatch(host):
    from cca_zoo_b200.deep import objectives as ours

    trials = F.loss_trials(SEED, TRIALS)
    assert len(trials) == len(G.META_LIVE["loss_fuzz"]) == 200
    bad, compared = [], 0
    for i, (t, meta) in enumerate(zip(trials, G.META_LIVE["loss_fuzz"])):
        if not t["determined"]:
            assert meta is None
            continue
        r = dict(meta, grads=[{p: G.live(f"loss_fuzz/{i}/{j}/{p}") for p in ("scale", "vals", "tr")}
                              for j in range(len(t["zs"]))] if meta["exc"] is None else None)
        msg = F.loss_mismatch(r, F.loss_record(ours, t, i), t)
        compared += 1
        if msg:
            bad.append(msg)
    assert compared > 50 and not bad, "\n".join(bad)
