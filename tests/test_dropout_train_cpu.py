"""CPU-side checks of train-mode dropout on the fused training paths (NAIS_basic / NAIS_regionEmbedding, model.py:71,162): the
segmented layout and `nais_train_users_dropout` take it as argument checks (nothing is launched, no GPU here), the host replay of
the cell-indexed mask, and the batched seed draw `model.train_users` relies on."""
import ctypes as C

import numpy as np
import torch

from poi_recommendation_models_b200 import _lib, ops

ERR_NULL, ERR_WORKSPACE, ERR_MODE = -1, -4, -5


def _one_branch_params(D=64, hid=64):
    """NAIS_regionEmbedding-shaped parameters with dropout 0.5 (pointers are never dereferenced: the argument checks run first)."""
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.beta = 1, hid, 1000, 10, _lib.DIST_NONE, 0.5
    br = p.branch[0]
    br.w_poi, br.w_reg = D // 2, D // 2
    br.hist_poi = br.tgt_poi = br.hist_reg = br.tgt_reg = 16
    br.w1, br.b1, br.w2 = 16, 16, 16
    p.dropout_p, p.dropout_seed = 0.5, 1234
    return p


def _segmented_batch():
    b = _lib.NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg = 16, 16, 16, 16
    b.B, b.n_seg, b.n_tiles, b.n_cells = 10, 1, 1, 50
    b.seg_offsets, b.row_offsets, b.seg_cell_offsets, b.tile_seg, b.tile_row0 = 16, 16, 16, 16, 16
    return b


def _states():
    o, d = _lib.NaisAdagrad(), _lib.NaisDenseAdagrad()
    for f in ("sum_w1", "sum_b1", "sum_w2"):
        setattr(d, f, 16)
    return o, d


def test_segmented_layout_accepts_one_branch_dropout():
    """The segmented layout takes dropout for one branch: a train step with a too-small workspace gets as far as the workspace
    check (it was NAIS_ERR_MODE).  Two branches (the disentangled model has no dropout) stay NAIS_ERR_MODE."""
    lib = _lib.load()
    p, b = _one_branch_params(), _segmented_batch()
    o, d = _states()
    assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 5, None) == ERR_WORKSPACE
    g = _lib.NaisGrads()
    assert lib.nais_pairs_backward_adagrad(C.byref(p), C.byref(b), 16, 16, None, 16, C.byref(g), C.byref(o), 16, 5, None) == ERR_WORKSPACE
    # two branches: the disentangled layout
    p2 = _one_branch_params()
    p2.n_branch = 2
    b0, b1 = p2.branch[0], p2.branch[1]
    b0.w_poi, b0.w_reg, b0.hist_reg, b0.tgt_reg = 64, 0, None, None
    b1.w_poi, b1.w_reg, b1.hist_reg, b1.tgt_reg, b1.w1, b1.b1, b1.w2 = 0, 64, 16, 16, 16, 16, 16
    for f in ("sum_region_w1", "sum_region_b1", "sum_region_w2"):
        setattr(d, f, 16)
    assert lib.nais_pairs_train_step(C.byref(p2), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 5, None) == ERR_MODE
    p2.dropout_p = 0.0
    assert lib.nais_pairs_train_step(C.byref(p2), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 5, None) == ERR_WORKSPACE


def test_train_users_dropout_needs_seeds_and_the_old_entries_refuse_dropout():
    lib = _lib.load()
    p = _one_branch_params()
    o, d = _states()
    indptr, users = np.array([0, 3, 5], dtype=np.int64), np.array([1, 0], dtype=np.int64)
    seeds = np.array([7, 8], dtype=np.uint64)
    common = (indptr.ctypes.data, 2, 16, 16, None, 16, None, users.ctypes.data, 2, 4, 0, C.byref(o), C.byref(d), 16, 16)
    assert lib.nais_train_users_dropout(C.byref(p), *common, 5, 0.0, 0.0, None, None) == ERR_NULL
    assert lib.nais_train_users_dropout(C.byref(p), *common, 5, 0.0, 0.0, seeds.ctypes.data, None) == ERR_WORKSPACE  # past the checks
    assert lib.nais_train_users(C.byref(p), *common, 5, None) == ERR_MODE
    assert lib.nais_train_users_centred(C.byref(p), *common, 5, 0.0, 0.0, None) == ERR_MODE
    # without dropout the seed array is not read, and the old entries behave as before
    p.dropout_p = 0.0
    assert lib.nais_train_users_dropout(C.byref(p), *common, 5, 0.0, 0.0, None, None) == ERR_WORKSPACE
    assert lib.nais_train_users(C.byref(p), *common, 5, None) == ERR_WORKSPACE
    assert lib.nais_train_users_centred(C.byref(p), *common, 5, 0.0, 0.0, None) == ERR_WORKSPACE


def test_cell_indexed_keep_mask_is_the_dense_mask_reshaped():
    B, H, hid, seed = 7, 13, 48, 2 ** 61 + 12345
    for p in (0.5, 0.1, 0.9):
        dense = ops.dropout_keep_mask(seed, B, H, hid, p)
        cells = ops.dropout_keep_mask_cells(seed, B * H, hid, p)
        assert cells.shape == (B * H, hid) and np.array_equal(cells.reshape(B, H, hid), dense)
        assert abs(cells.mean() - (1 - p)) < 0.03
    # element (cell, k) hashes seed + (cell * hid + k) * golden: cells c0.. are the replay of a seed advanced by c0 * hid steps
    c0, golden = 25, 0x9E3779B97F4A7C15
    shifted = (seed + c0 * hid * golden) % 2 ** 64
    assert np.array_equal(ops.dropout_keep_mask_cells(seed, 40, hid, 0.5)[c0:], ops.dropout_keep_mask_cells(shifted, 40 - c0, hid, 0.5))


def test_batched_seed_draw_equals_single_draws():
    """`model.train_users` draws its per-step dropout seeds as one `torch.randint(0, 2**62, (n,))`; the per-user loop of
    `fused_adagrad_step` draws them one `(1,)` at a time.  Torch's CPU generator gives the same values."""
    torch.manual_seed(2024)
    batched = torch.randint(0, 2 ** 62, (2000,))
    torch.manual_seed(2024)
    single = torch.cat([torch.randint(0, 2 ** 62, (1,)) for _ in range(2000)])
    assert torch.equal(batched, single)
