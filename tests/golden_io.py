"""Load the committed reference outputs (tests/golden) and rebuild their seeded inputs."""
from __future__ import annotations

import json
import os

import numpy as np

from cca_zoo_b200.datasets import conftest_views, joint_data

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

with open(os.path.join(_DIR, "reference_outputs.json")) as _f:
    META = json.load(_f)
_NPZ = np.load(os.path.join(_DIR, "reference_outputs.npz"))

CASES = {c["name"]: c for c in META["cases"]}
LOSS_CASES = {c["name"]: c for c in META["loss_cases"]}


def dataset(name, dtype="f64"):
    kind, args = (META["datasets"].get(name) or META_EXT["datasets"][name])
    if kind == "derived":     # oracle/make_golden_ext.py: a base data set, shifted and / or with a duplicated column
        views = [v.copy() for v in dataset(args["base"])]
        if "shift" in args:
            views = [v + args["shift"] for v in views]
        if "dup" in args:
            j, col = args["dup"]
            views[j] = np.hstack([views[j], views[j][:, col:col + 1]])
    else:
        views = conftest_views(args["name"]) if kind == "conftest" else joint_data(**args)
    if dtype == "f32":
        views = [v.astype(np.float32) for v in views]
    return views


def case_inputs(name):
    c = CASES[name]
    return dataset(c["dataset"], c["dtype"])


def case_outputs(name):
    m = len(META["datasets"][CASES[name]["dataset"]][1].get("n_features", [])) or None
    ws, mus, i = [], [], 0
    while f"{name}/w{i}" in _NPZ:
        ws.append(_NPZ[f"{name}/w{i}"])
        mus.append(_NPZ[f"{name}/mean{i}"])
        i += 1
    return ws, mus, _NPZ[f"{name}/score"]


def get(key):
    return _NPZ[key]


def loss_inputs(name):
    """Same recipe as oracle/make_golden.py:loss_inputs (torch CPU generator)."""
    import torch

    c = LOSS_CASES.get(name) or GLOSS_CASES[name]
    g = torch.Generator().manual_seed(c["seed"])
    zl = torch.randn(c["batch"], 4, generator=g, dtype=torch.float64)
    out = []
    for w in c["widths"]:
        a = torch.randn(4, w, generator=g, dtype=torch.float64)
        out.append(zl @ a + 0.5 * torch.randn(c["batch"], w, generator=g, dtype=torch.float64))
    return out


def loss_outputs(name):
    npz = _NPZ if name in LOSS_CASES else _NPZ_EXT
    grads, i = [], 0
    while f"{name}/grad{i}" in npz:
        grads.append(npz[f"{name}/grad{i}"])
        i += 1
    return float(npz[f"{name}/loss"]), grads


# ---- extension fixtures: estimators that call the MCCA core with extra fit arguments (make_golden_ext.py) ----
with open(os.path.join(_DIR, "reference_outputs_ext.json")) as _f:
    META_EXT = json.load(_f)
_NPZ_EXT = np.load(os.path.join(_DIR, "reference_outputs_ext.npz"))
PARTIAL_CASES = {c["name"]: c for c in META_EXT["partial_cases"]}
GROUP_CASES = {c["name"]: c for c in META_EXT["group_cases"]}
GLOSS_CASES = {c["name"]: c for c in META_EXT["gloss_cases"]}
CENTER_CASES = {c["name"]: c for c in META_EXT["center_cases"]}


def ext_inputs(name):
    """(views, extra): extra = confound matrix (PartialCCA cases) or per-view group labels (GRCCA cases); the same
    seeded recipes as oracle/make_golden_ext.py."""
    c = PARTIAL_CASES.get(name) or GROUP_CASES.get(name) or CENTER_CASES[name]
    views = dataset(c["dataset"], c["dtype"])
    if name in CENTER_CASES:
        return views, None
    rng = np.random.default_rng(c["seed"])
    if name in PARTIAL_CASES:
        extra = rng.standard_normal((views[0].shape[0], c["q"])) + np.linspace(0.3, 1.2, c["q"])
    else:
        extra = [rng.integers(0, g, size=v.shape[1]) for v, g in zip(views, c["n_groups"])]
    return views, extra


def ext_outputs(name):
    out, i = {"w": [], "mean": [], "beta": []}, 0
    while f"{name}/w{i}" in _NPZ_EXT:
        out["w"].append(_NPZ_EXT[f"{name}/w{i}"])
        out["mean"].append(_NPZ_EXT[f"{name}/mean{i}"])
        if f"{name}/beta{i}" in _NPZ_EXT:
            out["beta"].append(_NPZ_EXT[f"{name}/beta{i}"])
        i += 1
    out["score"] = _NPZ_EXT[f"{name}/score"]
    if f"{name}/partial_corr" in _NPZ_EXT:
        out["partial_corr"] = _NPZ_EXT[f"{name}/partial_corr"]
    return out


# ---- BASELINE config 3: CCALoss / MCCALoss at batch 4096 (oracle/make_golden_cfg3.py) ----
with open(os.path.join(_DIR, "reference_outputs_cfg3.json")) as _f:
    META_CFG3 = json.load(_f)
_NPZ_CFG3 = np.load(os.path.join(_DIR, "reference_outputs_cfg3.npz"))
CFG3_CASES = {c["name"]: c for c in META_CFG3["cases"]}


def cfg3_inputs(name):
    """Same recipe as oracle/make_golden_cfg3.py:cfg3_inputs (16 shared latents + unit noise, torch CPU generator)."""
    import torch

    c = CFG3_CASES[name]
    g = torch.Generator().manual_seed(c["seed"])
    zl = torch.randn(c["batch"], 16, generator=g, dtype=torch.float64)
    out = []
    for w in c["widths"]:
        a = torch.randn(16, w, generator=g, dtype=torch.float64)
        out.append(zl @ a + torch.randn(c["batch"], w, generator=g, dtype=torch.float64))
    return out


def cfg3_outputs(name):
    """(loss, [per-view dict(rows, fro, tr, c)]): sub-sampled rows, Frobenius norm and two probe projections."""
    grads, i = [], 0
    while f"{name}/grad{i}_rows" in _NPZ_CFG3:
        grads.append({k: _NPZ_CFG3[f"{name}/grad{i}_{k}"] for k in ("rows", "fro", "tr", "c")})
        i += 1
    return float(_NPZ_CFG3[f"{name}/loss"]), grads


def cfg3_check_gradient(g, ref, view_index, case, tol):
    """Compare a full gradient (numpy, float64) with the stored digest of the reference's gradient."""
    stride = META_CFG3["row_stride"]
    rng = np.random.default_rng(10_000 + case["seed"] + view_index)
    r, c = rng.standard_normal(g.shape[0]), rng.standard_normal(g.shape[1])
    scale = np.abs(ref["rows"]).max()
    e_rows = np.abs(g[::stride] - ref["rows"]).max() / scale
    e_fro = abs(np.linalg.norm(g) - float(ref["fro"])) / float(ref["fro"])
    e_tr = np.abs(g.T @ r - ref["tr"]).max() / np.abs(ref["tr"]).max()
    e_c = np.abs(g @ c - ref["c"]).max() / np.abs(ref["c"]).max()
    assert e_rows < tol, f"sampled rows differ: {e_rows:.2e}"
    assert e_fro < tol, f"Frobenius norm differs: {e_fro:.2e}"
    assert e_tr < tol, f"batch projection differs: {e_tr:.2e}"
    assert e_c < tol, f"width projection differs: {e_c:.2e}"
    return max(e_rows, e_fro, e_tr, e_c)


# ---- outputs of the live reference for the oracle, fuzz and drop-in tests (oracle/make_golden_live.py) ----
with open(os.path.join(_DIR, "reference_live.json")) as _f:
    META_LIVE = json.load(_f)
with np.load(os.path.join(_DIR, "reference_live.npz")) as _z:
    _LIVE = {k: _z[k] for k in _z.files}
_LIVE_INDEX = json.loads(bytes(_LIVE.pop("index")))


def live(key):
    """One stored array (the file holds one flat array per dtype; the index gives dtype, start and shape)."""
    dt, start, shape = _LIVE_INDEX[key]
    return _LIVE[dt][start:start + int(np.prod(shape))].reshape(shape)


def live_list(key):
    out = []
    while f"{key}/{len(out)}" in _LIVE_INDEX:
        out.append(live(f"{key}/{len(out)}"))
    return out


def sha256_matches(arrays, digests):
    """Same dtype, shape and bytes as the arrays the stored SHA-256 digests were taken of."""
    import hashlib

    got = [[str(a.dtype), list(a.shape), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()]
           for a in arrays]
    return got == digests
