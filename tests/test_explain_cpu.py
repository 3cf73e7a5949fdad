"""Explanations of pair scores without a GPU: the C entry points are declared and bound, every argument error is returned before
any launch, and the float64 per-item terms the GPU tests check against restate the oracle's score."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import explain_terms
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_NULL, ERR_SHAPE, ERR_WORKSPACE, ERR_MODE = -1, -2, -4, -5  # NAIS_ERR_* of include/nais_b200.h
NEW = ("nais_pairs_explain_workspace_bytes", "nais_pairs_explain")


def test_symbols_declared_and_bound():
    header = open(os.path.join(ROOT, "include", "nais_b200.h")).read()
    for name in NEW:
        assert re.search(r"NAIS_API\s+\w+\s+" + name + r"\s*\(", header), name
        assert name in _lib.SYMBOLS
    lib = _lib.load()
    for name in NEW:
        fn = getattr(lib, name)
        assert fn.restype == _lib.SYMBOLS[name][0] and list(fn.argtypes) == list(_lib.SYMBOLS[name][1])


def _params(dropout_p=0.0, n_branch=1):
    """NAIS_regionEmbedding-shaped (or disentangled-shaped) parameters: pointers are never dereferenced, the checks run first."""
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.beta = n_branch, 64, 1000, 10, _lib.DIST_NONE, 0.5
    for bi in range(n_branch):
        br = p.branch[bi]
        br.w_poi, br.w_reg = (32, 32) if n_branch == 1 else ((64, 0) if bi == 0 else (0, 64))
        br.hist_poi = br.tgt_poi = br.hist_reg = br.tgt_reg = 16
        br.w1, br.b1, br.w2 = 16, 16, 16
    p.dropout_p, p.dropout_seed = dropout_p, 1
    return p


def _dense(B=6, H=5):
    b = _lib.NaisPairs()
    b.hist = b.tgt = b.hreg = b.treg = 16
    b.B, b.H = B, H
    return b


def _segmented():
    b = _lib.NaisPairs()
    b.hist = b.tgt = b.hreg = b.treg = 16
    b.B, b.n_seg, b.n_tiles, b.n_cells = 7, 2, 2, 31
    b.seg_offsets = b.row_offsets = b.seg_cell_offsets = b.tile_seg = b.tile_row0 = 16
    return b


@pytest.mark.parametrize("layout", ["dense", "segmented"])
@pytest.mark.parametrize("n_branch", [1, 2])
def test_argument_errors_before_any_launch(layout, n_branch):
    lib = _lib.load()
    b = _dense() if layout == "dense" else _segmented()
    p = _params(n_branch=n_branch)
    cells = b.B * b.H if layout == "dense" else b.n_cells
    need = lib.nais_pairs_explain_workspace_bytes(C.byref(p), C.byref(b))
    assert need >= 4 * (2 * n_branch * cells + n_branch * b.B + b.B)  # cell_e, cell_es, row_sum, score
    launches = lib.nais_launch_count()

    def call(p=p, m=5, pos=16, contrib=16, ws=16, ws_bytes=need):
        return lib.nais_pairs_explain(C.byref(p), C.byref(b), m, None, pos, contrib, None, ws, ws_bytes, None)

    assert call(m=0) == ERR_SHAPE and call(m=33) == ERR_SHAPE and call(m=-1) == ERR_SHAPE
    assert call(p=_params(0.5, n_branch)) == ERR_MODE  # dropout: explanations are inference
    assert call(pos=None) == ERR_NULL and call(contrib=None) == ERR_NULL
    assert call(ws_bytes=need - 1) == ERR_WORKSPACE and call(ws_bytes=0) == ERR_WORKSPACE
    assert lib.nais_launch_count() == launches, "an argument error launched a kernel"


VARIANT_ARGS = {"basic": (False, None), "region": (True, None), "region_distance": (True, "latlon"), "distance": (False, "latlon"),
                "disentangled": (True, "km")}


@pytest.mark.parametrize("variant", list(VARIANT_ARGS))
def test_attention_terms_restate_the_oracle(variant):
    N, D, hid, B, H, beta = 50, 16, 12, 9, 7, 0.6
    rng = np.random.default_rng(3)
    coords, region = rng.uniform(-1, 1, (N, 2)) + [40.7, -74.0], rng.integers(0, 6, N)
    sd = orc.init_state(variant, N, D, hid, 6, 1, seed=4, style="trained")
    hist = np.stack([rng.choice(N, H, replace=False) for _ in range(B)])
    tgt = rng.integers(0, N, B)
    tgt[::3] = hist[::3, 2]  # training-style rows: the target inside its history
    reg, dist = VARIANT_ARGS[variant]
    aux = None
    if dist == "latlon":
        aux = torch.from_numpy(orc.latlon_abs_diff(coords, tgt, hist))
    elif dist == "km":
        aux = torch.from_numpy(orc.dist_km(coords[tgt][:, None, 0], coords[tgt][:, None, 1], coords[hist][..., 0], coords[hist][..., 1]))
    t = torch.from_numpy
    args = (t(hist), t(tgt), t(region[hist]) if reg else None, t(region[tgt]) if reg else None, aux)
    T = explain_terms.attention_terms(sd, variant, beta, *args)
    ref = orc.attention_network(sd, variant, beta, *args, dtype=torch.float64)
    assert torch.allclose(T["contrib"].sum(-1), ref, rtol=1e-12, atol=1e-12)
    assert torch.allclose(T["attn"].sum(-1), torch.ones_like(T["S"]), rtol=0, atol=1e-12)
    assert T["E"].shape[0] == (2 if variant == "disentangled" else 1)
    assert not T["E"][:, ~T["mask"]].any() and not T["contrib"][~T["mask"]].any()
    assert (T["E"][:, T["mask"]] > 0).all()
