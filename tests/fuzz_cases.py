"""Seeded differential-fuzz trials of the host logic of the estimators and the objectives.

Each trial draws its inputs from generators seeded once per run, runs one library (the reference or this package)
and reduces what that returns to a record of exactly the quantities that are compared; ``linear_mismatch`` and
``loss_mismatch`` check this package's record against the reference's.  tools/fuzz_vs_reference.py and
tools/fuzz_loss_vs_reference.py take the reference's records from the live reference; the suite takes them from
tests/golden/reference_live.{json,npz} (written by oracle/make_golden_live.py from the same seeds).
"""
from __future__ import annotations

import warnings

import numpy as np
import torch

from oracle import restatement as R


def _exc_name(e):
    return f"{type(e).__module__}.{type(e).__qualname__}"


# ---- estimators: random shapes, ridge values, centring flags, view weights, confounds, feature groups, dtypes ----
def linear_trials(seed, trials, medium=False):
    """The trial list of one seed.  Ill-posed draws (c = 0 with a rank-deficient or under-determined view, where the
    reference itself returns noise-dependent output) carry ``well=False``; only their exception type is compared."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(trials):
        model = str(rng.choice(["CCA", "rCCA", "PLS", "MCCA", "GCCA", "PartialCCA", "GRCCA"]))
        m = 2 if model in ("CCA", "rCCA", "PLS") else int(rng.integers(2, 5))
        n = int(rng.integers(6, 120))
        dims = [int(rng.integers(1, 30)) for _ in range(m)]
        k = int(rng.integers(1, 8))
        if medium:                          # wider views, explicit solver routes (top-k route needs 4k <= width)
            n = int(rng.integers(300, 700))
            dims = [int(rng.integers(36, 110)) for _ in range(m)]
        lat = rng.standard_normal((n, 3))
        views = [lat @ rng.standard_normal((3, d)) * rng.uniform(0, 1.5) + rng.standard_normal((n, d))
                 + rng.uniform(-1, 1) for d in dims]
        dup = rng.random() < 0.15
        if dup:
            j = int(rng.integers(0, m))
            views[j] = np.hstack([views[j], views[j][:, :1]])
            dims[j] += 1
        f32 = rng.random() < 0.25
        if f32:
            views = [v.astype(np.float32) for v in views]
        kw = dict(latent_dimensions=k, center=bool(rng.random() < 0.75))
        c = 0.0
        if model not in ("CCA", "PLS"):
            c = float(rng.choice([0.0, 0.0, 0.1, 0.5, 1.0])) if rng.random() < 0.7 else \
                [float(rng.uniform(0, 1)) for _ in range(m)]
            kw["c"] = c
        extra = {}
        ours_kw = {}
        if medium and model not in ("CCA", "PLS"):
            ours_kw["solver"] = str(rng.choice(["auto", "eigen", "cholesky"]))
        if model == "GCCA" and rng.random() < 0.5:
            kw["view_weights"] = [float(rng.uniform(0.5, 2)) for _ in range(m)]
        if model == "MCCA":
            kw["pca"] = bool(rng.random() < 0.5)
        if model == "PartialCCA":
            extra["partials"] = rng.standard_normal((n, int(rng.integers(1, 4)))) + 0.3
        if model == "GRCCA":
            kw["mu"] = float(rng.choice([0.0, 0.5, 2.0]))
            extra["feature_groups"] = [rng.integers(0, 3, size=d) for d in dims]
        cmin = 1.0 if model == "PLS" else (min(c) if isinstance(c, list) else c)
        q = extra["partials"].shape[1] if "partials" in extra else 0
        determined = (not dup) and n - 2 - q > sum(dims)     # else exact correlation-1 ties (degenerate top eigenspace)
        # c = 0 needs full-rank blocks; GCCA takes pinv(view) whatever c is; float32 inputs of an under-determined
        # problem amplify the reference's own float32 rounding (centring and pinv run in float32 there)
        well = determined or (cmin > 0 and model != "GCCA" and not f32)
        out.append(dict(model=model, n=n, dims=dims, q=q, f32=f32, views=views, kw=kw, extra=extra, ours_kw=ours_kw,
                        well=well, desc=f"{'well ' if well else 'ILL  '}{model} n={n} dims={dims} f32={f32} {kw} "
                                        f"{ours_kw}"))
    return out


def linear_record(lib, t, ours=False):
    """Fit ``t`` with ``lib`` (a module with the estimator classes) and keep what ``linear_mismatch`` compares."""
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            est = getattr(lib, t["model"])(**t["kw"], **(t["ours_kw"] if ours else {})).fit(t["views"], **t["extra"])
            held = [v[: t["n"] // 2] for v in t["views"]]
            score, tr, pair = est.score(t["views"]), est.transform(held), est.pairwise_correlations(held)
    except Exception as e:  # noqa: BLE001
        return {"exc": _exc_name(e)}
    return {"exc": None, "weights": [np.asarray(w) for w in est.weights_], "means": [np.asarray(m) for m in est.means_],
            "score": np.asarray(score), "pairwise": np.asarray(pair),
            "shapes": [list(w.shape) for w in est.weights_],
            "dtypes": [str(w.dtype) for w in est.weights_] + [str(np.asarray(x).dtype) for x in tr]}


def _determined(t, score):
    """Components whose weights and variates are compared: inside the rank of the problem, clearly correlated, and
    separated from both neighbours."""
    kmax = min(min(t["dims"]), max(t["n"] - 2 - t["q"], 0))
    left = np.abs(np.diff(np.concatenate([[2.0], score])))
    right = np.abs(np.diff(np.concatenate([score, [-2.0]])))
    return (left > 1e-3) & (right > 1e-3) & (np.abs(score) > 1e-3) & (np.arange(score.shape[0]) < kmax)


def linear_reduce(r, t):
    """The reference's record cut to what ``linear_mismatch`` reads of it: weights and pairwise correlations of the
    determined components only."""
    if r["exc"]:
        return r
    simple = _determined(t, r["score"])
    return dict(r, weights=[w[:, simple] for w in r["weights"]], pairwise=r["pairwise"][..., simple])


def linear_mismatch(r, o, t, show_all=False):
    """None if this package's record ``o`` agrees with the reference's reduced record ``r`` on trial ``t``, else
    what differs."""
    desc = t["desc"]
    if r["exc"] or o["exc"]:
        return None if r["exc"] == o["exc"] else f"EXCEPTION {desc} | ref: {r['exc']} | ours: {o['exc']}"
    if not t["well"] and not show_all:
        return None
    if r["shapes"] != o["shapes"]:
        return f"WEIGHT SHAPES {desc} {r['shapes']} {o['shapes']}"
    if r["dtypes"] != o["dtypes"]:
        return f"DTYPES {desc} {r['dtypes']} {o['dtypes']}"
    tol = 2e-3 if t["f32"] else 1e-6
    sc = r["score"]
    kmax = min(min(t["dims"]), max(t["n"] - 2 - t["q"], 0))
    d_score = float(np.max(np.abs(sc - o["score"])[np.arange(sc.shape[0]) < max(kmax, 1)]))
    # weights / variates of the determined components only (sign-aligned per component)
    simple = _determined(t, sc)
    w_r = [np.asarray(w, dtype=np.float64) for w in r["weights"]]
    w_o = R.align_signs([np.asarray(w, dtype=np.float64)[:, simple] for w in o["weights"]], w_r)
    d_w = 0.0
    for a, b in zip(w_o, w_r):
        num = np.linalg.norm(a - b, axis=0)
        den = np.linalg.norm(b, axis=0)
        if num.size:
            d_w = max(d_w, float(np.max(num / np.maximum(den, 1e-300))))
    d_means = max(float(np.max(np.abs(np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64))))
                  for a, b in zip(r["means"], o["means"]))
    d_pair = float(np.max(np.abs(r["pairwise"] - o["pairwise"][..., simple]))) if simple.any() else 0.0
    if not (d_score < tol and d_w < 50 * tol and d_means < 1e-5 and d_pair < 50 * tol):
        return f"VALUES score {d_score:.1e} weights {d_w:.1e} means {d_means:.1e} pairwise {d_pair:.1e} {desc}"
    return None


# ---- objectives: route selection and the analytic backward against the reference's forward + autograd ----
def loss_trials(seed, trials):
    """The trial list of one seed.  Batches with n - 1 <= 1.25 width (rank-deficient or barely determined batch
    covariance, where the reference differentiates through repeated eigenvalues and its own gradient is rounding
    noise) carry ``determined=False``."""
    g = torch.Generator().manual_seed(seed)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(trials):
        kind = str(rng.choice(["CCALoss", "MCCALoss", "GCCALoss"]))
        m = 2 if kind == "CCALoss" else int(rng.integers(2, 5))
        n = int(rng.integers(4, 200))
        widths = [int(rng.integers(1, 80)) for _ in range(m)]
        if kind == "GCCALoss" or rng.random() < 0.5:
            widths = [widths[0]] * m
        eps = float(rng.choice([1e-3, 1e-4, 1e-5]))
        dt = torch.float64 if rng.random() < 0.7 else torch.float32
        lat = torch.randn(n, 3, generator=g, dtype=torch.float64)
        zs = [(lat @ torch.randn(3, w, generator=g, dtype=torch.float64) * float(rng.uniform(0, 1.5))
               + torch.randn(n, w, generator=g, dtype=torch.float64)).to(dt) for w in widths]
        deficient = n - 1 <= 1.25 * (sum(widths) if kind == "GCCALoss" else max(widths))
        out.append(dict(kind=kind, eps=eps, dt=dt, zs=zs, determined=not deficient,
                        desc=f"{kind} n={n} widths={widths} eps={eps} {dt}"))
    return out


def grad_digest(g, salt):
    """A gradient reduced to its largest magnitude, 16 entries at seeded positions and its product with a seeded
    random vector over the batch (every entry of the gradient enters that product)."""
    rng = np.random.default_rng(salt)
    idx = rng.choice(g.size, min(g.size, 16), replace=False)
    return {"scale": np.abs(g).max().reshape(1), "vals": g.ravel()[idx], "tr": g.T @ rng.standard_normal(g.shape[0])}


def loss_record(lib, t, salt):
    """Forward + backward of trial ``t`` with ``lib`` (a module with the loss classes); ``salt`` seeds the digest."""
    zz = [z.clone().requires_grad_(True) for z in t["zs"]]
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            loss = getattr(lib, t["kind"])(eps=t["eps"])(zz)
            loss.backward()
    except Exception as e:  # noqa: BLE001
        return {"exc": _exc_name(e)}
    return {"exc": None, "loss": loss.item(), "dtype": str(loss.dtype), "dim": loss.dim(),
            "grads": [grad_digest(z.grad.double().numpy(), 1000 * salt + i) for i, z in enumerate(zz)]}


def loss_mismatch(r, o, t):
    """None if this package's record ``o`` agrees with the reference's ``r`` on trial ``t``, else what differs."""
    desc = t["desc"]
    if r["exc"] or o["exc"]:
        return None if r["exc"] == o["exc"] else f"EXCEPTION {desc} | ref {r['exc']} | ours {o['exc']}"
    tol = 5e-3 if t["dt"] == torch.float32 else 1e-7
    dl = abs(r["loss"] - o["loss"]) / max(abs(r["loss"]), 1e-300)
    dg = 0.0
    for a, b in zip(r["grads"], o["grads"]):
        scale = max(float(a["scale"][0]), 1e-300)
        dg = max(dg, np.abs(a["vals"] - b["vals"]).max() / scale, abs(float(a["scale"][0] - b["scale"][0])) / scale,
                 np.abs(a["tr"] - b["tr"]).max() / max(np.abs(a["tr"]).max(), 1e-300))
    if not (dl < tol and dg < 50 * tol) or (r["dtype"], r["dim"]) != (o["dtype"], o["dim"]):
        return f"VALUES loss {dl:.1e} grad {dg:.1e} dtype/dim {r['dtype'], r['dim']} {o['dtype'], o['dim']} {desc}"
    return None
