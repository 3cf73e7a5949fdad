"""CPU-side checks of the disentangled model on the tcgen05 pair kernels: the training step's workspace holds one ReLU pattern per
branch, the same [n_branch, cells] act_mask ops allocates, and the argument checks of the two-branch entry points are
unchanged (nothing is launched, no GPU here)."""
import ctypes as C

from poi_recommendation_models_b200 import _lib, ops


def _params(n_branch, D=64, hid=64):
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_buckets = n_branch, hid, 1000, 10, 1
    p.dist_mode = _lib.DIST_KM if n_branch == 2 else _lib.DIST_NONE
    p.dist_embed = 16
    b0, b1 = p.branch[0], p.branch[1]
    b0.w_poi, b0.w_reg, b0.hist_poi, b0.tgt_poi = D, 0, 16, 16
    b1.w_poi, b1.w_reg, b1.hist_reg, b1.tgt_reg = 0, D, 16, 16
    for br in (b0, b1):
        br.w1, br.b1, br.w2 = 16, 16, 16  # (never dereferenced)
    return p


def _dense(B, H):
    b = _lib.NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg, b.aux = 16, 16, 16, 16, 16
    b.B, b.H = B, H
    return b


def _segmented(B, n_cells):
    b = _lib.NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg = 16, 16, 16, 16
    b.B, b.n_seg, b.n_tiles, b.n_cells = B, 1, 1, n_cells
    b.seg_offsets, b.row_offsets, b.seg_cell_offsets, b.tile_seg, b.tile_row0 = 16, 16, 16, 16, 16
    b.hist_coords, b.tgt_coords = 16, 16
    return b


def test_act_mask_is_one_pattern_per_branch_in_ops_and_in_the_train_step():
    """ops allocates act_mask as [n_branch, cells], and the one-call training step's workspace holds the same: one more history
    item per row adds B cells, and the step's own buffers (the rest of the growth is the backward's workspace) grow by the
    words ops allocates for them, 8 bytes each."""
    lib = _lib.load()
    B = 32  # (B * 8 bytes per branch: whole 256-byte blocks, so the growth is exact)
    for n_branch in (1, 2):
        p = _params(n_branch)
        assert ops.act_mask_words(p, _dense(B, 20)) == n_branch * B * 20
        assert ops.act_mask_words(p, _segmented(B, 777)) == n_branch * 777
        growth = []
        for H in (20, 21):
            b = _dense(B, H)
            step = lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b))
            bwd = lib.nais_pairs_backward_workspace_bytes(C.byref(p), C.byref(b))
            assert step > bwd > 0
            growth.append(step - bwd)
        words = ops.act_mask_words(p, _dense(B, 21)) - ops.act_mask_words(p, _dense(B, 20))
        assert growth[1] - growth[0] == 8 * words == n_branch * B * 8, (n_branch, growth)


def test_two_branch_argument_errors_are_unchanged():
    lib = _lib.load()
    p = _params(2)
    b = _dense(8, 5)
    g = _lib.NaisGrads()
    # the presorting forward stays one-branch
    assert lib.nais_pairs_forward_presort(C.byref(p), C.byref(b), C.byref(g), 16, 16, 16, 16, 16, 1 << 20, None) == -5
    # NULL score / NULL km tensor / NULL embed_distance
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), None, None, None, None, None) == -1
    b.aux = None
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), 16, None, None, None, None) == -1
    b.aux = 16
    p.dist_embed = None
    assert lib.nais_pairs_forward(C.byref(p), C.byref(b), 16, None, None, None, None) == -1
    p.dist_embed = 16
    # two branches that are not the disentangled layout: the fused optimizer rejects them
    p.branch[1].w_poi, p.branch[1].w_reg, p.branch[1].hist_poi, p.branch[1].tgt_poi = 32, 32, 16, 16
    assert lib.nais_pairs_train_step_workspace_bytes(C.byref(p), C.byref(b)) == 0
