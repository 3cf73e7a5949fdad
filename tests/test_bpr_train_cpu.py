"""CPU-side checks of BPR training (nais_pairs_train_step_bpr / nais_train_users_bpr): the symbols are declared and bound, the
NaisBprLoss mirror has the header's layout, every argument error is returned before anything is launched (fake pointers: no GPU
here), and a float64 restatement of the loss and dL/dscore the kernel implements equals torch's autograd of -logsigmoid."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from poi_recommendation_models_b200 import _lib

ERR_NULL, ERR_SHAPE, ERR_WORKSPACE, ERR_MODE = -1, -2, -4, -5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRIES = ("nais_pairs_train_step_bpr", "nais_train_users_bpr")


def test_bpr_symbols_are_declared_and_bound():
    hdr = open(os.path.join(ROOT, "include", "nais_b200.h")).read()
    lib = _lib.load()
    for name in ENTRIES:
        assert re.search(r"NAIS_API int " + name + r"\(", hdr), name
        assert name in _lib.SYMBOLS and getattr(lib, name).argtypes == _lib.SYMBOLS[name][1], name
    # the BPR calls take the arguments of their BCE twins, the label / row_weight pair replaced by the loss descriptor
    assert _lib.SYMBOLS["nais_train_users_bpr"] == _lib.SYMBOLS["nais_train_users_dropout"]
    bce = _lib.SYMBOLS["nais_pairs_train_step"][1]
    assert _lib.SYMBOLS["nais_pairs_train_step_bpr"][1] == bce[:2] + [C.POINTER(_lib.NaisBprLoss)] + bce[4:]


def test_bpr_loss_mirror_matches_the_header_layout(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    fields = [f for f, _ in _lib.NaisBprLoss._fields_]
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "nais_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(NaisBprLoss));']
    lines += [f'  printf("{f} %zu\\n", offsetof(NaisBprLoss, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "bpr_layout.c", tmp_path / "bpr_layout"
    src.write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{os.path.join(ROOT, 'include')}", str(src), "-o", str(exe)], check=True)
    got = dict(ln.split() for ln in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert fields == ["num_neg", "reserved0", "group_weight"]
    assert int(got["size"]) == C.sizeof(_lib.NaisBprLoss) == 16
    for f in fields:
        assert int(got[f]) == getattr(_lib.NaisBprLoss, f).offset, f


def _params(dropout_p=0.0):
    """NAIS_regionEmbedding-shaped parameters (pointers are never dereferenced: the argument checks run first)."""
    p = _lib.NaisParams()
    p.n_branch, p.hid, p.item_num, p.region_num, p.dist_mode, p.beta = 1, 64, 1000, 10, _lib.DIST_NONE, 0.5
    br = p.branch[0]
    br.w_poi, br.w_reg = 32, 32
    br.hist_poi = br.tgt_poi = br.hist_reg = br.tgt_reg = 16
    br.w1, br.b1, br.w2 = 16, 16, 16
    p.dropout_p, p.dropout_seed = dropout_p, 1234
    return p


def _dense_batch(B=10, H=5):
    b = _lib.NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg, b.B, b.H = 16, 16, 16, 16, B, H
    return b


def _states():
    o, d = _lib.NaisAdagrad(), _lib.NaisDenseAdagrad()
    for f in ("sum_w1", "sum_b1", "sum_w2"):
        setattr(d, f, 16)
    return o, d


def test_train_step_bpr_argument_errors_come_before_any_launch():
    lib = _lib.load()
    p, o, d = _params(), *_states()

    def step(b, bpr, p=p, loss=16, ws=16, o=o, d=d):
        return lib.nais_pairs_train_step_bpr(C.byref(p), C.byref(b), None if bpr is None else C.byref(bpr), None if o is None else C.byref(o),
                                             None if d is None else C.byref(d), loss, None, ws, 5, None)

    ok = _lib.NaisBprLoss(4, 0, None)
    assert step(_dense_batch(10), ok) == ERR_WORKSPACE  # a valid call gets as far as the workspace size
    assert step(_dense_batch(10), _lib.NaisBprLoss(1, 0, 16)) == ERR_WORKSPACE
    assert step(_dense_batch(10), None) == ERR_NULL
    for nn in (0, -1):
        assert step(_dense_batch(10), _lib.NaisBprLoss(nn, 0, None)) == ERR_SHAPE
    assert step(_dense_batch(10), _lib.NaisBprLoss(3, 0, None)) == ERR_SHAPE  # 10 rows are not groups of 4
    assert step(_dense_batch(10), ok, loss=None) == ERR_NULL
    assert step(_dense_batch(10), ok, o=None) == ERR_NULL
    assert step(_dense_batch(10), ok, ws=None) == ERR_NULL
    assert step(_dense_batch(10), ok, ws=8) == -3  # NAIS_ERR_ALIGN
    assert step(_dense_batch(0), ok, ws=None) == 0  # nothing to do
    bad = _params()
    bad.hid = 0
    assert step(_dense_batch(10), ok, p=bad) == ERR_SHAPE
    b = _dense_batch(10)
    b.hreg = None
    assert step(b, ok) == ERR_NULL
    d2 = _lib.NaisDenseAdagrad()
    assert step(_dense_batch(10), ok, d=d2) == ERR_NULL


def test_train_users_bpr_argument_errors_come_before_any_launch():
    lib = _lib.load()
    p, o, d = _params(), *_states()
    indptr, users = np.array([0, 3, 5], dtype=np.int64), np.array([1, 0], dtype=np.int64)
    seeds = np.array([7, 8], dtype=np.uint64)

    def call(p, num_ng, seeds_ptr, ws=16):
        return lib.nais_train_users_bpr(C.byref(p), indptr.ctypes.data, 2, 16, 16, None, 16, None, users.ctypes.data, 2, num_ng, 0,
                                        C.byref(o), C.byref(d), 16, ws, 5, 0.0, 0.0, seeds_ptr, None)

    assert call(p, 4, None) == ERR_WORKSPACE  # past the checks
    assert call(p, 1, None) == ERR_WORKSPACE
    assert call(p, 0, None) == ERR_SHAPE  # BPR needs a negative per positive (BCE takes num_ng = 0)
    assert call(p, -1, None) == ERR_SHAPE
    assert call(p, 4, None, ws=None) == ERR_NULL
    pd = _params(dropout_p=0.5)
    assert call(pd, 4, None) == ERR_NULL  # dropout without seeds
    assert call(pd, 4, seeds.ctypes.data) == ERR_WORKSPACE
    users[0] = 2  # outside the CSR
    assert call(p, 4, None) == ERR_SHAPE
    users[0] = 1


def bpr_reference(s, num_neg, group_weight=None):
    """The kernel's contract in float64: (loss, dL/dscore) of sum_g w_g sum_j softplus(-(s[gG] - s[gG + j]))."""
    s = np.asarray(s, dtype=np.float64).reshape(-1, num_neg + 1)
    n_groups = s.shape[0]
    w = np.full(n_groups, 1.0 / (n_groups * num_neg)) if group_weight is None else np.asarray(group_weight, dtype=np.float64)
    d = s[:, :1] - s[:, 1:]
    loss = float((w[:, None] * (np.maximum(-d, 0.0) + np.log1p(np.exp(-np.abs(d))))).sum())
    z = np.exp(-np.abs(d))
    sig = np.where(d >= 0, z / (1 + z), 1 - z / (1 + z))  # sigma(-d), in torch's log_sigmoid backward form
    ds = np.empty_like(s)
    ds[:, 1:] = w[:, None] * sig
    ds[:, 0] = -ds[:, 1:].sum(axis=1)
    return loss, ds.reshape(-1)


@pytest.mark.parametrize("num_neg", [1, 4])
def test_float64_restatement_equals_torch_autograd(num_neg):
    rng = np.random.default_rng(num_neg)
    n_groups = 257
    s = rng.normal(size=n_groups * (num_neg + 1)) * 3
    s[: 10 * (num_neg + 1)] = rng.uniform(-200, 200, size=10 * (num_neg + 1))  # saturated: |d| up to 400
    w = rng.uniform(0.1, 1.0, size=n_groups)
    for gw in (None, w):
        t = torch.tensor(s, dtype=torch.float64, requires_grad=True)
        v = t.view(-1, num_neg + 1)
        nll = -torch.nn.functional.logsigmoid(v[:, 0:1] - v[:, 1:])
        loss = nll.mean() if gw is None else (nll * torch.tensor(gw)[:, None]).sum()
        loss.backward()
        loss = float(loss.detach())
        ref_loss, ref_ds = bpr_reference(s, num_neg, gw)
        assert np.isfinite(ref_loss) and np.isfinite(ref_ds).all()
        assert abs(ref_loss - loss) <= 1e-12 * abs(loss), (ref_loss, loss)
        np.testing.assert_allclose(ref_ds, t.grad.numpy(), rtol=1e-12, atol=1e-300)
