"""CPU-side checks of the disentangled model's training paths: the two-branch rule of the fused optimizer entry points and the
segmented layout's NAIS_DIST_KM requirements are argument checks (nothing is launched, no GPU here), and `dist_km_pairs` is
powerLaw.dist."""
import ctypes as C

import numpy as np

import nais_testutil as util
from oracle import nais_oracle as orc
from poi_recommendation_models_b200 import _lib, batches as PB


def _disentangled_params(D=64, hid=64):
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.dist_buckets = 2, hid, 1000, 10, _lib.DIST_KM, 1
    p.dist_embed = 16
    b0, b1 = p.branch[0], p.branch[1]
    b0.w_poi, b0.w_reg, b0.hist_poi, b0.tgt_poi = D, 0, 16, 16
    b1.w_poi, b1.w_reg, b1.hist_reg, b1.tgt_reg = 0, D, 16, 16
    for br in (b0, b1):
        br.w1, br.b1, br.w2 = 16, 16, 16  # (never dereferenced: the argument checks run first)
    return p


def _segmented_batch():
    b = _lib.NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg = 16, 16, 16, 16
    b.B, b.n_seg, b.n_tiles, b.n_cells = 10, 1, 1, 50
    b.seg_offsets, b.row_offsets, b.seg_cell_offsets, b.tile_seg, b.tile_row0 = 16, 16, 16, 16, 16
    b.hist_coords, b.tgt_coords = 16, 16
    return b


def _full_dense_state():
    d = _lib.NaisDenseAdagrad()
    for f in ("sum_w1", "sum_b1", "sum_w2", "sum_region_w1", "sum_region_b1", "sum_region_w2", "sum_dist_embed"):
        setattr(d, f, 16)
    return d


def test_segmented_km_needs_coordinates():
    lib = _lib.load()
    p = _disentangled_params()
    b = _segmented_batch()
    b.hist_coords = None
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), 16, None, None, None, None) == -1
    b.hist_coords, b.tgt_coords = 16, None
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), 16, None, None, None, None) == -1
    p.dropout_p = 0.5  # segmented-layout dropout stays rejected
    b.tgt_coords = 16
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), 16, None, None, None, None) == -5


def test_two_branches_sharing_a_poi_part_are_rejected():
    """Both branches with a POI part: one sparse step per branch would step the shared tables twice -> NAIS_ERR_MODE."""
    lib = _lib.load()
    p = _disentangled_params()
    p.branch[1].w_poi, p.branch[1].w_reg = 32, 32
    p.branch[1].hist_poi = p.branch[1].tgt_poi = 16
    b = _segmented_batch()
    g, o, d = _lib.NaisGrads(), _lib.NaisAdagrad(), _full_dense_state()
    assert lib.nais_pairs_backward_adagrad(C.byref(p), C.byref(b), 16, 16, None, 16, C.byref(g), C.byref(o), 16, 1 << 30, None) == -5
    assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 1 << 30, None) == -5
    indptr, users = np.array([0, 3, 5], dtype=np.int64), np.array([1], dtype=np.int64)
    assert lib.nais_train_users(C.byref(p), indptr.ctypes.data, 2, 16, 16, 16, 16, 16, users.ctypes.data, 1, 4, 0, C.byref(o),
                                C.byref(d), 16, 16, 1 << 30, None) == -5
    assert lib.nais_train_users_centred(C.byref(p), indptr.ctypes.data, 2, 16, 16, 16, 16, 16, users.ctypes.data, 1, 4, 0, C.byref(o),
                                        C.byref(d), 16, 16, 1 << 30, 40.0, -74.0, None) == -5
    assert lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b)) == 0
    assert lib.nais_train_users_workspace_bytes(C.byref(p), 100, 4) == 0


def test_disentangled_layout_needs_the_new_dense_sums():
    lib = _lib.load()
    p = _disentangled_params()
    b = _segmented_batch()
    o = _lib.NaisAdagrad()
    indptr, users = np.array([0, 3, 5], dtype=np.int64), np.array([1], dtype=np.int64)
    for missing in ("sum_region_w1", "sum_region_b1", "sum_region_w2", "sum_dist_embed"):
        d = _full_dense_state()
        setattr(d, missing, None)
        assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 1 << 30, None) == -1, missing
        assert lib.nais_train_users_centred(C.byref(p), indptr.ctypes.data, 2, 16, 16, 16, 16, 16, users.ctypes.data, 1, 4, 0, C.byref(o),
                                            C.byref(d), 16, 16, 1 << 30, 0.0, 0.0, None) == -1, missing
    # without the distance term embed_distance is not a parameter of the step
    p.dist_mode = _lib.DIST_NONE
    d = _full_dense_state()
    d.sum_dist_embed = None
    assert lib.nais_pairs_train_step(C.byref(p), C.byref(b), 16, None, C.byref(o), C.byref(d), 16, None, 16, 5, None) == -4  # past the state checks
    # the lat/lon distance lanes are no two-branch layout of the fused paths
    p.dist_mode, p.dist_w, p.dist_b = _lib.DIST_LATLON, 16, 16
    g = _lib.NaisGrads()
    assert lib.nais_pairs_backward_adagrad(C.byref(p), C.byref(b), 16, 16, None, 16, C.byref(g), C.byref(o), 16, 1 << 30, None) == -5


def test_disentangled_workspace_queries():
    lib = _lib.load()
    p = _disentangled_params()
    b = _segmented_batch()
    one = lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b))
    assert one > lib.nais_pairs_backward_workspace_bytes(C.byref(p), C.byref(b)) > 0
    assert lib.nais_train_users_workspace_bytes(C.byref(p), 100, 4) > 0
    p.dist_mode = _lib.DIST_NONE
    assert lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b)) > 0


def test_dist_km_pairs_is_powerlaw_dist():
    z = util.load_golden("geo.npz")
    a, b = z["a"], z["b"]
    coords = np.concatenate([a, b])  # targets are rows 0..63, histories rows 64..127
    n = len(a)
    km = PB.dist_km_pairs(coords, np.arange(n), np.arange(n, 2 * n)[:, None], device="cpu").numpy()
    assert km.shape == (n, 1) and km.dtype == np.float32
    np.testing.assert_allclose(km[:, 0], z["dist"].astype(np.float32), rtol=1e-12, atol=0)
    # a [H] history broadcast to every target, against the oracle's float64 values
    rng = np.random.default_rng(0)
    c = np.stack([40.6 + rng.random(50) * 0.3, -74.1 + rng.random(50) * 0.3], 1)
    tgt, hist = rng.integers(0, 50, 7), rng.integers(0, 50, 11)
    got = PB.dist_km_pairs(c, tgt, hist, device="cpu").numpy()
    ref = orc.dist_km(c[tgt][:, None, 0], c[tgt][:, None, 1], c[hist][None, :, 0], c[hist][None, :, 1])
    np.testing.assert_allclose(got, ref.astype(np.float32), rtol=1e-12, atol=0)
    assert (got[np.equal.outer(tgt, hist)] == 0).all()

