"""Generate tests/golden/reference_live.{npz,json} from the UNMODIFIED reference: what the tests that once needed
the live reference compare against.

    python oracle/make_golden_live.py

TEST INFRASTRUCTURE ONLY (see make_golden.py).  Three groups of outputs:
  * oracle: the reference estimators on the reference's conftest fixtures, and SHA-256 digests of what the JointData
    generator and the conftest fixtures draw (tests/test_oracle_vs_reference.py pins oracle/restatement.py and
    cca_zoo_b200.datasets against them);
  * fuzz: the reference's records of the seeded fuzz trials of tests/fuzz_cases.py (tests/test_fuzz_vs_reference.py);
  * dropin: the reference's own GridSearchCV over its own estimators (tests/test_dropin_vs_reference.py).
The fuzz records are stored in float32 except the canonical correlations: the rounding (6e-8 relative) is below 1/50
of the tolerance of every comparison that reads them (5e-5 relative on weights, gradients and pairwise correlations,
1e-5 absolute on means).
"""
from __future__ import annotations

import hashlib
import importlib.util
import json
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import fuzz_cases as F  # noqa: E402  (before refshim: the reference has its own `tests` package)
from oracle import refshim  # noqa: E402

refshim.install()

import cca_zoo.linear as ref_linear  # noqa: E402
from cca_zoo.datasets import JointData  # noqa: E402
from cca_zoo.deep import objectives as ref_objectives  # noqa: E402
from cca_zoo.linear import GCCA, GRCCA, MCCA, PartialCCA, rCCA  # noqa: E402
from cca_zoo.model_selection import GridSearchCV  # noqa: E402

from cca_zoo_b200.datasets import conftest_views  # noqa: E402

FUZZ_SEED, FUZZ_TRIALS = 20240924, 200
JOINT_ARGS = dict(n_views=3, n_samples=77, latent_dimensions=3, n_features=[5, 9, 4],
                  signal_to_noise=[0.5, 1.0, 2.0], random_state=11)
CONFTEST = ["two_views", "three_views", "correlated_views", "two_views_test"]
RCCA = [(ds, c) for ds in ["two_views", "correlated_views"] for c in [0.0, 0.1, [0.2, 0.7], 1.0]]
MCCA_CASES = [(0.0, True), (0.0, False), (0.3, False), ([0.1, 0.2, 0.3], True)]
GCCA_CASES = [(0.0, None), (0.2, [1.0, 1.0, 2.0])]
PARTIAL = [(0.0, True, 2), (0.2, True, 3), ([0.1, 0.3], False, 2)]
GROUPED = [(0.0, 0.0, 2), (0.5, 0.0, 2), ([0.3, 0.6, 0.0], [0.5, 2.0, 1.0], 3)]
CENTER = ["MCCA", "MCCA_pca", "GCCA", "GCCA_w"]
DROPIN = [("rCCA", 2, {"c": [0.0, 0.1, 0.5, 0.9]}), ("MCCA", 3, {"c": [0.0, 0.3], "eps": [1e-6, 1e-3]}),
          ("GCCA", 3, {"c": [0.1, 0.6]})]


def dropin_views():
    """The 150-sample three-view draw the drop-in test searches over (rebuilt by the test)."""
    rng = np.random.default_rng(0)
    lat = rng.standard_normal((150, 2))
    return [lat @ rng.standard_normal((2, 8)) + rng.standard_normal((150, 8)),
            lat @ rng.standard_normal((2, 6)) + rng.standard_normal((150, 6)),
            lat @ rng.standard_normal((2, 5)) + rng.standard_normal((150, 5))]


def put_list(out, key, arrays, dtype=None):
    for i, a in enumerate(arrays):
        out[f"{key}/{i}"] = np.asarray(a, dtype=dtype)


def sha256(arrays):
    return [[str(a.dtype), list(a.shape), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()]
            for a in arrays]


def oracle_outputs(out, meta):
    for ds, c in RCCA:
        v = conftest_views(ds)
        est = rCCA(latent_dimensions=3, c=c).fit(v)
        put_list(out, f"rcca/{ds}/{c}/w", est.weights_)
        out[f"rcca/{ds}/{c}/score"] = est.score(v)
    for c, pca in MCCA_CASES:
        put_list(out, f"mcca/{c}/{pca}/w", MCCA(latent_dimensions=3, c=c, pca=pca).fit(conftest_views("three_views"))
                 .weights_)
    for c, mu in GCCA_CASES:
        put_list(out, f"gcca/{c}/{mu}/w", GCCA(latent_dimensions=3, c=c, view_weights=mu)
                 .fit(conftest_views("three_views")).weights_)
    meta["joint_data"] = sha256(JointData(**JOINT_ARGS).sample())
    spec = importlib.util.spec_from_file_location("ref_conftest", os.path.join(refshim.REFERENCE_ROOT, "tests",
                                                                               "conftest.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for name in CONFTEST:
        meta["conftest"][name] = sha256(getattr(mod, name).__wrapped__())
    for c, center, nv in PARTIAL:
        v = conftest_views("three_views")[:nv]
        Z = np.random.default_rng(7).standard_normal((v[0].shape[0], 3)) + 0.7
        est = PartialCCA(latent_dimensions=2, c=c, center=center).fit(v, partials=Z)
        put_list(out, f"partialcca/{c}/{center}/{nv}/w", est.weights_)
        put_list(out, f"partialcca/{c}/{center}/{nv}/beta", est.confound_betas_)
    for c, mu, nv in GROUPED:
        v = conftest_views("three_views")[:nv]
        rng = np.random.default_rng(5)
        gs = [rng.integers(0, 3, size=x.shape[1]) for x in v]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            put_list(out, f"grcca/{c}/{mu}/{nv}/w", GRCCA(latent_dimensions=2, c=c, mu=mu).fit(v, feature_groups=gs)
                     .weights_)
    for model in CENTER:
        v = [x + 1.3 for x in conftest_views("three_views")]
        if model.startswith("MCCA"):
            est = MCCA(latent_dimensions=3, c=0.1, center=False, pca=model.endswith("pca")).fit(v)
        else:
            vw = [1.0, 2.0, 0.5] if model.endswith("w") else None
            est = GCCA(latent_dimensions=3, c=0.1, center=False, view_weights=vw).fit(v)
        put_list(out, f"center/{model}/w", est.weights_)
        put_list(out, f"center/{model}/mean", est.means_)
    v = conftest_views("two_views")
    put_list(out, "ridge_null/w", rCCA(latent_dimensions=9, c=0.2).fit([v[0], np.hstack([v[1], v[1][:, :1]])])
             .weights_)


def fuzz_outputs(out, meta):
    """Only what the comparison reads: values of the well-posed trials, the exception type of every trial."""
    for i, t in enumerate(F.linear_trials(FUZZ_SEED, FUZZ_TRIALS)):
        r = F.linear_reduce(F.linear_record(ref_linear, t), t)
        meta["fuzz"].append({k: r[k] for k in ("exc", "shapes", "dtypes") if k in r and (t["well"] or k == "exc")})
        if r["exc"] is None and t["well"]:
            put_list(out, f"fuzz/{i}/w", r["weights"], np.float32)
            put_list(out, f"fuzz/{i}/mean", r["means"], np.float32)
            out[f"fuzz/{i}/score"], out[f"fuzz/{i}/pairwise"] = r["score"], r["pairwise"].astype(np.float32)
    for i, t in enumerate(F.loss_trials(FUZZ_SEED, FUZZ_TRIALS)):
        if not t["determined"]:
            meta["loss_fuzz"].append(None)
            continue
        r = F.loss_record(ref_objectives, t, i)
        meta["loss_fuzz"].append({k: r[k] for k in ("exc", "loss", "dtype", "dim") if k in r})
        for j, g in enumerate(r.get("grads", [])):
            for p in ("scale", "vals", "tr"):
                out[f"loss_fuzz/{i}/{j}/{p}"] = g[p].astype(np.float32)


def dropin_outputs(out, meta):
    views = dropin_views()
    for name, nv, grid in DROPIN:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            gs = GridSearchCV(getattr(ref_linear, name)(latent_dimensions=2), param_grid=grid, cv=3).fit(views[:nv])
        out[f"dropin/{name}/mean_test_score"] = gs.cv_results_["mean_test_score"]
        params = [{k.split("__", 1)[1]: v for k, v in p.items()} for p in gs.cv_results_["params"]]  # estimator__c
        meta["dropin"][name] = {"params": params, "best_params": gs.best_params_}


def pack(out):
    """Thousands of small arrays as one flat array per dtype plus a JSON index {key: [dtype, start, shape]} (one
    zip member per array would cost more than the data)."""
    flat, index = {}, {}
    for key, a in out.items():
        a = np.asarray(a)
        parts = flat.setdefault(a.dtype.str, [])
        index[key] = [a.dtype.str, sum(x.size for x in parts), list(a.shape)]
        parts.append(a.ravel())
    packed = {dt: np.concatenate(parts) for dt, parts in flat.items()}
    packed["index"] = np.array(json.dumps(index, separators=(",", ":")).encode())
    return packed


def main():
    out, meta = {}, {"conftest": {}, "fuzz_seed": FUZZ_SEED, "fuzz_trials": FUZZ_TRIALS, "fuzz": [], "loss_fuzz": [],
                     "dropin": {}}
    oracle_outputs(out, meta)
    fuzz_outputs(out, meta)
    dropin_outputs(out, meta)
    gdir = os.path.join(ROOT, "tests", "golden")
    np.savez_compressed(os.path.join(gdir, "reference_live.npz"), **pack(out))
    with open(os.path.join(gdir, "reference_live.json"), "w") as f:
        json.dump(meta, f, separators=(",", ":"))
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    main()
