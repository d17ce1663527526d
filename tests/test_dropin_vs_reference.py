"""Drop-in check of the sklearn model-selection contract (clone / get_params / set_params / fit / score), host logic
on the torch-CPU stand-in: a 3-fold grid search over this package's estimators must give the mean test scores and
the best parameters that the reference's own GridSearchCV gives over the reference's estimators (stored in
tests/golden/reference_live.* by oracle/make_golden_live.py).  The folds are the reference's: sklearn's KFold(3) over
the rows, and a fold's score is the mean of the estimator's per-component scores."""
import numpy as np
import pytest
from sklearn.base import clone
from sklearn.model_selection import KFold, ParameterGrid

from tests import fake_ops
from tests import golden_io as G

GRIDS = [("rCCA", 2, {"c": [0.0, 0.1, 0.5, 0.9]}), ("MCCA", 3, {"c": [0.0, 0.3], "eps": [1e-6, 1e-3]}),
         ("GCCA", 3, {"c": [0.1, 0.6]})]


@pytest.fixture
def host(monkeypatch):
    fake_ops.install(monkeypatch)


def test_reference_gridsearch_drives_our_estimators(host):
    import warnings

    from cca_zoo_b200 import linear as ours

    rng = np.random.default_rng(0)
    lat = rng.standard_normal((150, 2))
    views = [lat @ rng.standard_normal((2, 8)) + rng.standard_normal((150, 8)),
             lat @ rng.standard_normal((2, 6)) + rng.standard_normal((150, 6)),
             lat @ rng.standard_normal((2, 5)) + rng.standard_normal((150, 5))]
    for name, nv, grid in GRIDS:
        ref = G.META_LIVE["dropin"][name]
        params = list(ParameterGrid(grid))
        assert params == ref["params"], name
        base = getattr(ours, name)(latent_dimensions=2)
        scores = []
        for p in params:
            fold = []
            for tr, te in KFold(3).split(views[0]):
                est = clone(clone(base).set_params(**p))
                assert est.get_params()["c"] == p["c"]
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    est.fit([v[tr] for v in views[:nv]])
                fold.append(float(np.mean(est.score([v[te] for v in views[:nv]]))))
            scores.append(np.mean(fold))
        best = params[int(np.argmax(scores))]
        assert best == ref["best_params"], (name, best, ref["best_params"])
        assert np.allclose(G.live(f"dropin/{name}/mean_test_score"), scores, atol=1e-8), (name, scores)
        refit = clone(base).set_params(**best).fit(views[:nv])
        assert type(refit).__module__.startswith("cca_zoo_b200")
