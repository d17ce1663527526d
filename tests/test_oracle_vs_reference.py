"""Pin the oracle against the reference's outputs (tests/golden/reference_live.*, made from the reference by
oracle/make_golden_live.py).

This is the evidence behind the "parity pinned" line in oracle/restatement.py: each ref_* / cov_* function against
the reference estimator it restates, on the reference's own conftest fixtures, plus the data generators.
"""
import numpy as np
import pytest

from oracle import restatement as R
from tests import golden_io as G

from cca_zoo_b200.datasets import conftest_views, joint_data


def _C(views, center=True):
    M, s, n = R.moments(views)
    return R.covariance_from_moments(M, s, n, center), n


@pytest.mark.parametrize("c", [0.0, 0.1, [0.2, 0.7], 1.0])
@pytest.mark.parametrize("ds", ["two_views", "correlated_views"])
def test_rcca(ds, c):
    v = conftest_views(ds)
    ref_w, ref_score = G.live_list(f"rcca/{ds}/{c}/w"), G.live(f"rcca/{ds}/{c}/score")
    w, mu = R.ref_rcca_fit(v, 3, c)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-12
    C, n = _C(v)
    w, _ = R.cov_rcca_fit(C, [10, 8], 3, c, n)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-9
    np.testing.assert_allclose(R.score(v, mu, w), ref_score, rtol=1e-9)


@pytest.mark.parametrize("c,pca", [(0.0, True), (0.0, False), (0.3, False), ([0.1, 0.2, 0.3], True)])
def test_mcca(c, pca):
    v = conftest_views("three_views")
    ref_w = G.live_list(f"mcca/{c}/{pca}/w")
    w, _ = R.ref_mcca_fit(v, 3, c)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-10
    C, n = _C(v)
    w, _ = R.cov_mcca_fit(C, [10, 8, 6], 3, c)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-10


@pytest.mark.parametrize("c,mu", [(0.0, None), (0.2, [1.0, 1.0, 2.0])])
def test_gcca(c, mu):
    v = conftest_views("three_views")
    ref_w = G.live_list(f"gcca/{c}/{mu}/w")
    w, _ = R.ref_gcca_fit(v, 3, c, mu)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-10
    C, n = _C(v)
    w, _ = R.cov_gcca_fit(C, [10, 8, 6], n, 3, c, mu)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-9


def test_joint_data_generator_matches_reference():
    """Bit for bit the draws of the reference's JointData(...).sample() with the same arguments."""
    args = dict(n_views=3, n_samples=77, latent_dimensions=3, n_features=[5, 9, 4],
                signal_to_noise=[0.5, 1.0, 2.0], random_state=11)
    assert G.sha256_matches(joint_data(**args), G.META_LIVE["joint_data"])


def test_conftest_fixture_recipe_matches_reference_file():
    """The fixture recipe in cca_zoo_b200.datasets must draw, bit for bit, the fixtures of the reference's
    tests/conftest.py."""
    for name in ["two_views", "three_views", "correlated_views", "two_views_test"]:
        assert G.sha256_matches(conftest_views(name), G.META_LIVE["conftest"][name]), name


@pytest.mark.parametrize("c,center,nv", [(0.0, True, 2), (0.2, True, 3), ([0.1, 0.3], False, 2)])
def test_partialcca(c, center, nv):
    v = conftest_views("three_views")[:nv]
    Z = np.random.default_rng(7).standard_normal((v[0].shape[0], 3)) + 0.7
    ref_w, ref_betas = G.live_list(f"partialcca/{c}/{center}/{nv}/w"), G.live_list(f"partialcca/{c}/{center}/{nv}/beta")
    w, _, betas = R.ref_partialcca_fit(v, Z, 2, c, center=center)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-12
    M, s, n = R.moments(v + [Z])
    w, betas = R.cov_partialcca(M, s, n, [x.shape[1] for x in v], 3, 2, c, center=center)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-9
    assert len(betas) == len(ref_betas)
    for a, b in zip(betas, ref_betas):
        np.testing.assert_allclose(a, b, atol=1e-12)


@pytest.mark.parametrize("c,mu,nv", [(0.0, 0.0, 2), (0.5, 0.0, 2), ([0.3, 0.6, 0.0], [0.5, 2.0, 1.0], 3)])
def test_grcca(c, mu, nv):
    v = conftest_views("three_views")[:nv]
    rng = np.random.default_rng(5)
    gs = [rng.integers(0, 3, size=x.shape[1]) for x in v]
    ref_w = G.live_list(f"grcca/{c}/{mu}/{nv}/w")
    w, _ = R.ref_grcca_fit(v, gs, 2, c, mu)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-10
    C, n = _C(v)
    w = R.cov_grcca(C, [x.shape[1] for x in v], gs, 2, c, mu)
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-9


@pytest.mark.parametrize("model", ["MCCA", "MCCA_pca", "GCCA", "GCCA_w"])
def test_center_false_semantics(model):
    """np.cov centres inside MCCA / GCCA even when ``center=False``; GCCA mixes in raw second moments."""
    v = [x + 1.3 for x in conftest_views("three_views")]
    M, s, n = R.moments(v)
    C, Cu = R.covariance_from_moments(M, s, n, True), R.covariance_from_moments(M, s, n, False)
    dims = [10, 8, 6]
    if model.startswith("MCCA"):
        w, _ = R.ref_mcca_fit(v, 3, 0.1, center=False)
        wc, _ = R.cov_mcca_fit(C, dims, 3, 0.1)
    else:
        vw = [1.0, 2.0, 0.5] if model.endswith("w") else None
        w, _ = R.ref_gcca_fit(v, 3, 0.1, vw, center=False)
        wc, _ = R.cov_gcca_fit(C, dims, n, 3, 0.1, vw, second_moment=Cu)
    ref_w, ref_means = G.live_list(f"center/{model}/w"), G.live_list(f"center/{model}/mean")
    assert R.max_rel_err_per_vector(w, ref_w) < 1e-9
    assert R.max_rel_err_per_vector(wc, ref_w) < 1e-8
    assert len(ref_means) == 3 and all(np.all(np.asarray(m) == 0) for m in ref_means)


def test_ridge_keeps_the_null_directions_of_a_rank_deficient_view():
    v = conftest_views("two_views")
    v = [v[0], np.hstack([v[1], v[1][:, :1]])]          # 9 columns of rank 8
    ref_w = G.live_list("ridge_null/w")
    assert ref_w[0].shape == (10, 9)                   # nothing dropped: (1-c) lam + c >= c
    C, n = _C(v)
    w, sv = R.cov_rcca_fit(C, [10, 9], 9, 0.2, n)
    assert w[0].shape == (10, 9) and sv[-1] < 1e-7     # the 9th singular value is the null direction
    assert R.max_rel_err_per_vector([x[:, :8] for x in w], [x[:, :8] for x in ref_w]) < 1e-9
