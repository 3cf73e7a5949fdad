"""Tensor-level wrappers over the C ABI (include/nais_b200.h).

PyTorch is plumbing here: it owns device memory, the current stream and autograd bookkeeping; every number is computed
by the CUDA kernels in libnais_b200.so.  All ops raise if the tensors are not on a CUDA device — there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import (DIST_KM, DIST_LATLON, DIST_NONE, PAIRS_PRECISIONS, PRECISIONS, NaisAdagrad, NaisBranch, NaisCatalog,
                   NaisDenseAdagrad, NaisGrads, NaisPairs, NaisParams, NaisUsers)

# Every parameter of a variant as (name, role, branch), in the reference's state_dict order (SURVEY.md §5 checkpoint row): autograd
# returns the gradients by this position.  The role names the slot of the C structs (include/nais_b200.h) on that branch:
#   "hist_poi" / "tgt_poi"  embedding table: NaisBranch.<role>, NaisGrads.<role>[branch], NaisAdagrad.sum_<role>[branch]
#   "reg"                   region table: NaisBranch.hist_reg and .tgt_reg, NaisGrads.reg[branch], NaisAdagrad.sum_reg[branch]
#   "w1" / "b1" / "w2"      attention MLP: NaisBranch.<role>, NaisGrads.<role>[branch], NaisDenseAdagrad.sum_<role> (branch 0)
#                           or sum_region_<role> (branch 1)
#   "dist_w" / "dist_b" / "dist_embed"  distance term, one for both branches: NaisParams / NaisGrads.<role>,
#                           NaisDenseAdagrad.sum_<role>
_HIST, _TGT = ("embed_history.weight", "hist_poi", 0), ("embed_target.weight", "tgt_poi", 0)
_MLP = (("attn_layer1.weight", "w1", 0), ("attn_layer1.bias", "b1", 0), ("attn_layer2.weight", "w2", 0))
_DIST_LAYER = (("dist_layer.weight", "dist_w", 0), ("dist_layer.bias", "dist_b", 0))
VARIANT_SLOTS: Dict[str, Tuple[Tuple[str, str, int], ...]] = {
    "basic": (_HIST, _TGT) + _MLP,
    "region": (_HIST, _TGT, ("embed_region.weight", "reg", 0)) + _MLP,
    # embed_distance.weight exists in this class but is never read by its forward (model.py:204,270-276)
    "region_distance": (_HIST, _TGT, ("embed_region.weight", "reg", 0)) + _MLP + _DIST_LAYER,
    "distance": (_HIST, _TGT) + _MLP + _DIST_LAYER,
    # branch 1 scores the region table with its own MLP; the reference only ever reads row 0 of embed_distance (model.py:497-498)
    "disentangled": (_HIST, _TGT, ("embed_region.weight", "reg", 1), ("embed_distance.weight", "dist_embed", 0)) + _MLP
                    + (("region_attn_layer1.weight", "w1", 1), ("region_attn_layer1.bias", "b1", 1), ("region_attn_layer2.weight", "w2", 1)),
}
_TABLE_ROLES = frozenset(("hist_poi", "tgt_poi", "reg"))
_SHARED_ROLES = frozenset(("dist_w", "dist_b", "dist_embed"))
VARIANT_PARAMS: Dict[str, Tuple[str, ...]] = {v: tuple(n for n, _, _ in s) for v, s in VARIANT_SLOTS.items()}
_TABLES = tuple(dict.fromkeys(n for s in VARIANT_SLOTS.values() for n, role, _ in s if role in _TABLE_ROLES))
# gradients param_reduce_kernel writes in full (csrc/nais_bwd.cu): no zero fill needed; every other tensor has rows / entries the
# backward does not touch (untouched table rows, the rows of embed_distance past row 0)
_FULLY_WRITTEN = {n for s in VARIANT_SLOTS.values() for n, role, _ in s if role in ("w1", "b1", "w2", "dist_w", "dist_b")}
_N_BRANCH = {v: 1 + max(bi for _, _, bi in s) for v, s in VARIANT_SLOTS.items()}
# the optimizer-state field of each parameter: (name, NaisAdagrad field, branch) of the tables, (name, NaisDenseAdagrad field, None)
# of the rest
_ADAGRAD_FIELDS = {(v, tables): tuple((n, "sum_" + role, bi) if tables else (n, ("sum_region_" if bi else "sum_") + role, None)
                                      for n, role, bi in s if (role in _TABLE_ROLES) == tables)
                   for v, s in VARIANT_SLOTS.items() for tables in (True, False)}
VARIANT_DIST = {"basic": (DIST_NONE, 0.0), "region": (DIST_NONE, 0.0), "region_distance": (DIST_LATLON, 100.0),
                "distance": (DIST_LATLON, 1000.0), "disentangled": (DIST_KM, 0.0)}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts) -> torch.device:
    dev = None
    flat = []
    for t in ts:  # a SegmentedPairs stands for all of its device arrays
        flat.extend(v for v in vars(t).values() if isinstance(v, torch.Tensor)) if isinstance(t, SegmentedPairs) else flat.append(t)
    for t in flat:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("NAIS ops run only on a CUDA device (no CPU fallback); got a tensor on " + str(t.device))
        dev = dev or t.device
        if t.device != dev:
            raise RuntimeError("NAIS ops: tensors on different devices")
    return dev


def _f32(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise RuntimeError("NAIS ops compute in float32; got " + str(t.dtype))
    return t.contiguous()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# ----------------------------------------------------------------------------------------------------------------------
# Out-of-range ids (nn.Embedding raises IndexError; the kernels cannot): every pair call enqueues a poll of the library's
# device-side bad-index word into pinned host memory (nais_poll_bad_index: an async 4-byte copy, no synchronisation) and
# looks at the polls that have completed since — so a bad id raises on a LATER call of this module, or at once with
# `check_indices(sync=True)`.  The kernels themselves never use such an id as an address (include/nais_b200.h).
# ----------------------------------------------------------------------------------------------------------------------
_POLL_SLOTS = 64
_POLLS: Dict[int, dict] = {}  # device index -> {"buf": pinned int32 [_POLL_SLOTS], "next": slot, "inflight": [(slot, event)]}


def _poll_state(dev: torch.device) -> dict:
    st = _POLLS.get(dev.index or 0)
    if st is None:
        st = {"buf": torch.zeros(_POLL_SLOTS, dtype=torch.int32).pin_memory(), "next": 0, "inflight": []}
        _POLLS[dev.index or 0] = st
    return st


_POLL_EVERY = 8  # a poll costs ~90 us of host time (event + pinned read): the word stays raised on the device, nothing is lost


def _poll_bad_index(dev: torch.device) -> None:
    if torch.cuda.is_current_stream_capturing():
        return  # inside a CUDA graph capture: the word stays raised on the device until the next poll outside a graph
    st = _poll_state(dev)
    st["calls"] = st.get("calls", 0) + 1
    if st["calls"] % _POLL_EVERY != 1 and _POLL_EVERY > 1:
        return
    check_indices(dev, sync=len(st["inflight"]) >= _POLL_SLOTS - 1)
    _enqueue_poll(st)


def _enqueue_poll(st: dict) -> None:
    """nais_poll_bad_index into the next pinned slot on the current stream, and an event that tells when the slot is valid."""
    slot = st["next"]
    st["next"] = (slot + 1) % _POLL_SLOTS
    _lib.check(_lib.load().nais_poll_bad_index(st["buf"].data_ptr() + 4 * slot, _stream()), "nais_poll_bad_index")
    ev = torch.cuda.Event()
    ev.record()
    st["inflight"].append((slot, ev))


def check_indices(dev=None, sync: bool = False) -> None:
    """Raise IndexError if a kernel enqueued before a completed poll met a POI / region id outside its table (what
    nn.Embedding raises in the reference).  `sync=True` first polls once more and waits for every poll in flight."""
    devs = list(_POLLS) if dev is None else [torch.device(dev).index or 0]
    bad = False
    for d in devs:
        st = _POLLS.get(d)
        if st is None:
            if not sync:
                continue
            st = _poll_state(torch.device("cuda", d))
        if sync and not torch.cuda.is_current_stream_capturing():
            with torch.cuda.device(d):
                _enqueue_poll(st)
        q = st["inflight"]
        while q and (sync or q[0][1].query()):
            slot, ev = q.pop(0)
            ev.synchronize()
            bad = bad or bool(st["buf"][slot].item())
            st["buf"][slot] = 0
    if bad:
        raise IndexError("index out of range in a NAIS id tensor (a POI or region id outside its embedding table; detected on "
                         "the device by an earlier kernel — no table row was read or written through it)")


def build_params(variant: str, P: Dict[str, torch.Tensor], beta: float, keep: List[torch.Tensor],
                 dropout_p: float = 0.0, dropout_seed: int = 0, pairs_precision: str = "auto") -> NaisParams:
    """NaisParams for a reference-shaped parameter dict.  Contiguous copies are appended to `keep` to stay alive.
    `pairs_precision`: "auto" (tcgen05 pair kernels where the shape has them), "fp32", "tc" (NAIS_PAIRS_*)."""
    p = NaisParams()
    mode, scale = VARIANT_DIST[variant]
    p.dist_mode, p.dist_scale, p.beta = mode, scale, float(beta)
    p.dist_buckets, p.dist_bucket_km, p.region_num, p.n_branch = 1, 1.0, 0, _N_BRANCH[variant]
    p.dropout_p, p.dropout_seed = float(dropout_p), int(dropout_seed)
    p.pairs_precision = PAIRS_PRECISIONS[pairs_precision]
    b0 = p.branch[0]
    b0_tensors = {}
    for name, role, bi in VARIANT_SLOTS[variant]:
        t = _f32(P[name].detach())
        keep.append(t)
        if role in _SHARED_ROLES:
            setattr(p, role, t.data_ptr())
            continue
        br = p.branch[1] if bi else b0
        if role == "reg":
            br.hist_reg = br.tgt_reg = t.data_ptr()
            br.w_reg, p.region_num = t.shape[1], t.shape[0]
        else:
            setattr(br, role, t.data_ptr())
        if bi == 0:
            b0_tensors[role] = t
    eh, w1, b1, w2 = b0_tensors["hist_poi"], b0_tensors["w1"], b0_tensors["b1"], b0_tensors["w2"]
    p.item_num, p.hid = eh.shape[0], w1.shape[0]
    b0.w_poi = eh.shape[1]
    w_in = b0.w_poi + b0.w_reg + (2 if mode == DIST_LATLON else 0)
    if w1.shape[1] != w_in or b1.numel() != p.hid or w2.numel() != p.hid:
        raise RuntimeError(f"attn_layer shapes do not match the variant: w1 {tuple(w1.shape)}, expected [*, {w_in}]")
    return p


def _grads_struct(variant: str, grads: Dict[str, int], remaps: Optional[Dict[str, int]] = None) -> NaisGrads:
    """NaisGrads with the slot of every parameter in `grads` (name -> device address of its gradient) set; every other slot stays
    NULL, so the backward skips it.  A table in `remaps` (name -> address of its int32 remap) gets row-compacted gradients:
    its `grads` entry is then the address of the touched rows (NaisGrads::remap_*)."""
    g = NaisGrads()
    for name, role, bi in VARIANT_SLOTS[variant]:
        ptr = grads.get(name)
        if ptr is None:
            continue
        if role in _SHARED_ROLES:
            setattr(g, role, ptr)
        else:
            getattr(g, role)[bi] = ptr
        if remaps and name in remaps:
            getattr(g, "remap_" + role)[bi] = remaps[name]
    return g


def _adagrad_struct(variant: str, P: Dict[str, torch.Tensor], sums: Dict[str, torch.Tensor], lr: float, eps: float, tables: bool):
    """NaisAdagrad of the embedding tables (`tables`) or NaisDenseAdagrad of the other parameters, from the optimizer's
    `state['sum']` of each (`sums`: name -> tensor).  (embed_distance: the kernels read and step row 0 only, so the state's
    row 0 — the start of the tensor — is what they get.)"""
    s = NaisAdagrad() if tables else NaisDenseAdagrad()
    s.lr, s.eps = float(lr), float(eps)
    for name, field, bi in _ADAGRAD_FIELDS[variant, tables]:
        st = sums[name]
        if st.dtype != torch.float32 or not st.is_contiguous() or st.shape != P[name].shape or not P[name].is_contiguous():
            raise RuntimeError(f"fused Adagrad: {name} and its state must be contiguous float32 of the same shape")
        if bi is None:
            setattr(s, field, st.data_ptr())
        else:
            getattr(s, field)[bi] = st.data_ptr()
    return s


@dataclass
class SegmentedPairs:
    """A multi-user training batch in the segmented layout of NaisPairs (include/nais_b200.h): the rows of a segment (= a
    user) share ONE stored history — no [B,H] repeat (batches.py:97), no materialised [B,H,2] distance tensor (run.py:239-247:
    the kernels form |dlat|,|dlon|, or the haversine km of the disentangled model, from centred coordinates; `center` is the
    (lat, lon) that was subtracted from them).  Built by `segment_structure` + `sample_batch`
    (batches.DeviceBatcher.multi_user_batch) or by hand."""
    hist: torch.Tensor                 # [nnz] int64 history POI ids, segment after segment
    hreg: Optional[torch.Tensor]       # [nnz] int64
    hist_coords: Optional[torch.Tensor]  # [nnz,2] float32 centred
    tgt: torch.Tensor                  # [B] int64
    treg: Optional[torch.Tensor]       # [B] int64
    tgt_coords: Optional[torch.Tensor]  # [B,2] float32 centred
    label: Optional[torch.Tensor]      # [B] float32
    seg_offsets: torch.Tensor          # [n_seg+1] int64 (device)
    row_offsets: torch.Tensor          # [n_seg+1] int64
    seg_cell_offsets: torch.Tensor     # [n_seg+1] int64
    tile_seg: torch.Tensor             # [n_tiles] int32
    tile_row0: torch.Tensor            # [n_tiles] int64
    n_seg: int
    B: int
    n_tiles: int
    n_cells: int
    max_hist: int
    host_row_offsets: Optional[object] = None  # numpy copy (per-user loss weights etc.)
    center: Tuple[float, float] = (0.0, 0.0)


def _upload_packed(arrays, device):
    """Several small host index arrays -> the device in ONE copy (a pageable host-to-device copy blocks the host for ~15 us;
    a one-user batch has five of them): everything rides in one int64 buffer, int32 arrays as a reinterpreted tail."""
    import numpy as np
    parts, spans = [], []
    off = 0
    for a, dt in arrays:
        a = np.ascontiguousarray(np.asarray(a).astype(dt))
        n64 = a.size if dt == np.int64 else (a.size + 1) // 2
        buf = np.zeros(n64, dtype=np.int64)
        buf.view(dt)[: a.size] = a
        parts.append(buf)
        spans.append((off, a.size, dt))
        off += n64
    dev_buf = torch.from_numpy(np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)).to(device)
    out = []
    for o, n, dt in spans:
        n64 = n if dt == np.int64 else (n + 1) // 2
        t = dev_buf[o:o + n64]
        out.append(t if dt == np.int64 else t.view(torch.int32)[:n])
    return out


def segment_structure(hist_lens, rows_per_seg, device, extra=()) -> Dict[str, object]:
    """Host-side structure of a segmented batch (numpy, O(segments + tiles)): offsets and the tile table the kernels walk.
    Tile t covers at most min(16, 128 // H_s) rows of ONE segment (1 row when H_s > 128; csrc/nais_pairs_tile.cuh).
    `extra`: more (array, dtype) pairs to ride in the same upload (returned under "extra")."""
    import numpy as np
    H = np.asarray(hist_lens, dtype=np.int64)
    R = np.asarray(rows_per_seg, dtype=np.int64)
    R = np.where(H > 0, R, 0)
    seg_off = np.concatenate([[0], np.cumsum(H)])
    row_off = np.concatenate([[0], np.cumsum(R)])
    cell_off = np.concatenate([[0], np.cumsum(R * H)])
    rpt = np.where(H > 0, np.minimum(16, np.maximum(1, 128 // np.maximum(H, 1))), 1)
    tiles = (R + rpt - 1) // rpt
    tile_seg = np.repeat(np.arange(len(H), dtype=np.int32), tiles)
    first = np.concatenate([[0], np.cumsum(tiles)])[:-1]
    within = np.arange(int(tiles.sum()), dtype=np.int64) - np.repeat(first, tiles)
    tile_row0 = np.repeat(row_off[:-1], tiles) + within * np.repeat(rpt, tiles)
    up = _upload_packed([(seg_off, np.int64), (row_off, np.int64), (cell_off, np.int64), (tile_row0, np.int64), (tile_seg, np.int32)]
                        + [(a, dt) for a, dt in extra], device)
    return dict(seg_offsets=up[0], row_offsets=up[1], seg_cell_offsets=up[2], tile_row0=up[3], tile_seg=up[4], n_seg=len(H),
                B=int(row_off[-1]), n_tiles=int(tiles.sum()), n_cells=int(cell_off[-1]), max_hist=int(H.max()) if len(H) else 0,
                host_row_offsets=row_off, host_seg_offsets=seg_off, extra=up[5:])


def sample_batch(hist: torch.Tensor, st: Dict[str, object], num_ng: int, item_num: int, seed: int,
                 poi_region: Optional[torch.Tensor] = None, poi_coords: Optional[torch.Tensor] = None):
    """nais_sample_batch: targets / labels / target regions / target coordinates of a segmented batch, sampled ON THE DEVICE
    (batches.py:67-108 for many users at once: positives + `num_ng` negatives each, uniform without replacement over the
    POIs outside the user's history).  `st` = `segment_structure(H_s, (num_ng + 1) * H_s)`."""
    dev = _need_cuda(hist, st["seg_offsets"], poi_region, poi_coords)
    B = st["B"]
    with torch.cuda.device(dev):
        tgt = torch.empty(B, dtype=torch.int64, device=dev)
        label = torch.empty(B, dtype=torch.float32, device=dev)
        treg = torch.empty(B, dtype=torch.int64, device=dev) if poi_region is not None else None
        tc = torch.empty(B, 2, dtype=torch.float32, device=dev) if poi_coords is not None else None
        pr = None if poi_region is None else poi_region.to(torch.int32).contiguous()
        pc = None if poi_coords is None else _f32(poi_coords)
        _lib.check(_lib.load().nais_sample_batch(st["seg_offsets"].data_ptr(), hist.data_ptr(), st["n_seg"], st["row_offsets"].data_ptr(),
                                                 int(num_ng), int(item_num), _ptr(pr), _ptr(pc), int(seed) & (2 ** 64 - 1), st["max_hist"],
                                                 tgt.data_ptr(), label.data_ptr(), _ptr(treg), _ptr(tc), _stream()), "nais_sample_batch")
    return tgt, label, treg, tc


def _pairs_struct(hist, tgt, hreg, treg, aux, keep) -> NaisPairs:
    if isinstance(hist, SegmentedPairs):
        sp = hist
        b = NaisPairs()
        b.hist, b.tgt, b.hreg, b.treg, b.aux = _ptr(sp.hist), _ptr(sp.tgt), _ptr(sp.hreg), _ptr(sp.treg), None
        b.B, b.H, b.n_seg = sp.B, 0, sp.n_seg
        b.seg_offsets, b.row_offsets, b.seg_cell_offsets = _ptr(sp.seg_offsets), _ptr(sp.row_offsets), _ptr(sp.seg_cell_offsets)
        b.tile_seg, b.tile_row0, b.n_tiles, b.n_cells = _ptr(sp.tile_seg), _ptr(sp.tile_row0), sp.n_tiles, sp.n_cells
        b.hist_coords, b.tgt_coords = _ptr(sp.hist_coords), _ptr(sp.tgt_coords)
        b.center_lat, b.center_lon = float(sp.center[0]), float(sp.center[1])
        keep.append(sp)
        return b

    def i64(t):
        if t is None:
            return None
        t = t.to(torch.int64).contiguous()
        keep.append(t)
        return t
    hist, tgt, hreg, treg = i64(hist), i64(tgt), i64(hreg), i64(treg)
    if hist.dim() != 2 or tgt.dim() != 1 or hist.shape[0] != tgt.shape[0]:
        raise RuntimeError(f"expected history [B,H] and target [B]; got {tuple(hist.shape)} and {tuple(tgt.shape)}")
    if aux is not None:
        aux = _f32(aux)
        keep.append(aux)
    b = NaisPairs()
    b.hist, b.tgt, b.hreg, b.treg, b.aux = _ptr(hist), _ptr(tgt), _ptr(hreg), _ptr(treg), _ptr(aux)
    b.B, b.H = hist.shape[0], hist.shape[1]
    return b


def pairs_dispatch(p: NaisParams, b: NaisPairs) -> Tuple[bool, bool]:
    """(forward on tcgen05?, backward on tcgen05?) for these parameters and this batch (nais_pairs_dispatch)."""
    f, g = C.c_int32(0), C.c_int32(0)
    _lib.check(_lib.load().nais_pairs_dispatch(C.byref(p), C.byref(b), C.byref(f), C.byref(g)), "nais_pairs_dispatch")
    return bool(f.value), bool(g.value)


# The autograd forward sorts the coming backward's id lists next to its own kernel (nais_pairs_forward_presort: the sorts depend on
# the batch only; -50 us of a C3-sized step).  The backward workspace then lives from forward to backward instead of inside the
# backward call; set to False to keep it transient (e.g. many forwards of large batches before the first backward).
PRESORT_IN_FORWARD = True


class _PairCall:
    """What every pair entry point of the library does around its call: the device guard, the NaisParams (and the NaisPairs of
    `batch` = (hist, tgt, hreg, treg, aux)) with their contiguous copies kept alive, the workspace, the return-code check and,
    once the call is enqueued, the bad-index poll.  `with _PairCall(...) as c: c.launch(entry, ...)`."""

    def __init__(self, dev: torch.device, variant: str, beta: float, P: Dict[str, torch.Tensor], precision: str, drop=(0.0, 0),
                 batch=None):
        self.dev, self.variant, self.lib, self.keep = dev, variant, _lib.load(), []
        self._guard = torch.cuda.device(dev)
        self._args = (beta, P, drop, precision, batch)

    def __enter__(self) -> "_PairCall":
        beta, P, drop, precision, batch = self._args
        self._guard.__enter__()
        try:
            self.p = build_params(self.variant, P, beta, self.keep, drop[0], drop[1], precision)
            self.b = None if batch is None else _pairs_struct(*batch, self.keep)
        except BaseException:
            self._guard.__exit__(None, None, None)
            raise
        self.structs = (C.byref(self.p),) if self.b is None else (C.byref(self.p), C.byref(self.b))
        return self

    def __exit__(self, exc_type, exc, tb) -> None:
        try:
            if exc_type is None:
                _poll_bad_index(self.dev)
        finally:
            self._guard.__exit__(exc_type, exc, tb)

    def query(self, entry: str, *args) -> int:
        """lib.<entry>(p[, b], *args): a workspace size."""
        return getattr(self.lib, entry)(*self.structs, *args)

    def launch(self, entry: str, *args, ws_bytes: Optional[int] = None, ws: Optional[torch.Tensor] = None, tail=()):
        """lib.<entry>(p[, b], *args[, workspace, ws_bytes], *tail, stream), raising on a non-zero return code.  A workspace of
        `ws_bytes` is allocated unless `ws` is given; returns it."""
        if ws_bytes is not None:
            ws = torch.empty(max(ws_bytes, 16), device=self.dev, dtype=torch.uint8) if ws is None else ws
            args += (ws.data_ptr(), ws_bytes)
        _lib.check(getattr(self.lib, entry)(*self.structs, *args, *tail, _stream()), entry)
        return ws


def act_mask_words(p: NaisParams, b: NaisPairs) -> int:
    """Words of the act_mask nais_pairs_forward writes for (p, b): [n_branch, cells] (include/nais_b200.h)."""
    return p.n_branch * (b.n_cells if b.seg_offsets else b.B * b.H)


def _forward_launch(c: _PairCall, want_mask: bool = True, presort: bool = False):
    """nais_pairs_forward -> (score, row_sum, parts, act_mask, presorted workspace): act_mask is the ReLU pattern the tcgen05
    forward saves for the tcgen05 backward (int64 [n_branch * cells], branch bi's from bi * cells; with dropout "active and
    kept"; None when the FP32 forward runs or hid > 64).  With `presort`
    (one-branch variants) the call is nais_pairs_forward_presort and the last element is the backward workspace holding the
    sorted id lists for nais_pairs_backward_presorted; else None."""
    p, b, dev = c.p, c.b, c.dev
    B = b.B
    score = torch.empty(B, device=dev, dtype=torch.float32)
    row_sum = torch.empty(p.n_branch, B, device=dev, dtype=torch.float32)
    parts = torch.empty(p.n_branch, B, device=dev, dtype=torch.float32)
    mask = None
    if want_mask and B and p.hid <= 64 and pairs_dispatch(p, b)[0]:
        mask = torch.empty(act_mask_words(p, b), device=dev, dtype=torch.int64)
    outs = (score.data_ptr(), row_sum.data_ptr(), parts.data_ptr(), _ptr(mask))
    # (the backward tiles exist for D, hid <= 128: a wider forward-only shape keeps the plain call)
    if presort and B and p.n_branch == 1 and p.hid <= 128 and p.branch[0].w_poi + p.branch[0].w_reg <= 128:
        ws_bytes = c.query("nais_pairs_backward_workspace_bytes")
        ws = torch.empty(max(ws_bytes, 16), device=dev, dtype=torch.uint8)
        # (the forward reads only which table slots are set: they tell it which id lists the coming backward reduces)
        g = _grads_struct(c.variant, {n: ws.data_ptr() for n in VARIANT_PARAMS[c.variant] if n in _TABLES})
        c.launch("nais_pairs_forward_presort", C.byref(g), *outs, ws_bytes=ws_bytes, ws=ws)
        return score, row_sum, parts, mask, ws
    c.launch("nais_pairs_forward", *outs)
    return score, row_sum, parts, mask, None


def _grad_buffers(P: Dict[str, torch.Tensor], n_rows: int, tables: bool) -> Dict[str, torch.Tensor]:
    """The dense float32 gradient of every parameter (`tables=False`: but the embedding tables) for a batch of `n_rows` rows."""
    def buf(name, t):
        mk = torch.empty_like if (name in _FULLY_WRITTEN and n_rows > 0) else torch.zeros_like  # (an empty batch launches nothing)
        return mk(t, dtype=torch.float32, memory_format=torch.contiguous_format)
    return {n: buf(n, t) for n, t in P.items() if tables or n not in _TABLES}


def _addresses(G: Dict[str, torch.Tensor]) -> Dict[str, int]:
    return {n: t.data_ptr() for n, t in G.items()}


def _fwd_bwd(pairs_precision):
    """`pairs_precision` is one name for both directions or a (forward, backward) pair."""
    return (pairs_precision, pairs_precision) if isinstance(pairs_precision, str) else tuple(pairs_precision)


class _PairsFunction(torch.autograd.Function):
    """score = attention_network(pairs).  forward -> nais_pairs_forward, backward -> nais_pairs_backward."""

    @staticmethod
    def forward(ctx, variant, beta, drop, hist, tgt, hreg, treg, aux, *params):
        names = VARIANT_PARAMS[variant]
        P = dict(zip(names, params))
        dev = _need_cuda(hist, tgt, hreg, treg, aux, *params)
        need_bwd = any(t.requires_grad for t in params) and (len(drop) < 4 or bool(drop[3]))  # drop[3]: grad mode at the call
        # (the forward and the backward must agree on the pair kernels' precision for the lists / workspace to match)
        presort = need_bwd and PRESORT_IN_FORWARD and _fwd_bwd(drop[2])[0] == _fwd_bwd(drop[2])[1]
        with _PairCall(dev, variant, beta, P, _fwd_bwd(drop[2])[0], drop, (hist, tgt, hreg, treg, aux)) as c:
            score, row_sum, parts, mask, ws = _forward_launch(c, want_mask=need_bwd, presort=presort)
        ctx.presorted_ws = ws  # (not an input or an output: rides on ctx; used once)
        ctx.variant, ctx.beta, ctx.drop = variant, beta, drop
        ctx.seg = hist if isinstance(hist, SegmentedPairs) else None  # (not a tensor: rides on ctx)
        e = torch.empty(0)
        ctx.save_for_backward(e if ctx.seg is not None else hist, tgt if tgt is not None else e, hreg if hreg is not None else e,
                              treg if treg is not None else e, aux if aux is not None else e, row_sum, parts,
                              mask if mask is not None else e, *params)
        ctx.has = (hreg is not None, treg is not None, aux is not None, mask is not None)
        return score

    @staticmethod
    def backward(ctx, dscore):
        hist, tgt, hreg, treg, aux, row_sum, parts, mask, *params = ctx.saved_tensors
        if ctx.seg is not None:
            hist, tgt = ctx.seg, None
        hreg = hreg if ctx.has[0] else None
        treg = treg if ctx.has[1] else None
        aux = aux if ctx.has[2] else None
        mask = mask if ctx.has[3] else None
        names = VARIANT_PARAMS[ctx.variant]
        P = dict(zip(names, params))
        ws, ctx.presorted_ws = ctx.presorted_ws, None  # (a second backward through a retained graph sorts again)
        G = pairs_backward_raw(ctx.variant, ctx.beta, P, hist, tgt, hreg, treg, aux, row_sum, parts, dscore, ctx.drop, act_mask=mask,
                               presorted_ws=ws)
        grads = tuple(G[n].to(P[n].dtype) if ctx.needs_input_grad[8 + i] else None for i, n in enumerate(names))
        return (None, None, None, None, None, None, None, None) + grads


def pairs_backward_raw(variant: str, beta: float, P: Dict[str, torch.Tensor], hist, tgt, hreg, treg, aux, row_sum, parts, dscore,
                       drop=(0.0, 0, "auto"), tables: bool = True, act_mask: Optional[torch.Tensor] = None,
                       presorted_ws: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """nais_pairs_backward: every parameter gradient of `pairs_score` given dscore [B] and the forward's saved row sums / per-
    branch scores (/ ReLU pattern `act_mask`, when the tcgen05 forward produced one), as a dict of dense float32 tensors (zero
    rows for untouched table rows).  `tables=False` skips the embedding tables (no sort, no segment reduce): the attention-MLP /
    dist-layer gradients only.  `presorted_ws`: the workspace nais_pairs_forward_presort left for this batch (`tables=True`)."""
    dev = _need_cuda(hist, tgt, dscore, *P.values())
    with _PairCall(dev, variant, beta, P, _fwd_bwd(drop[2])[1], drop, (hist, tgt, hreg, treg, aux)) as c:
        G = _grad_buffers(P, int(c.b.B), tables)
        g = _grads_struct(variant, _addresses(G))
        ws_bytes = c.query("nais_pairs_backward_workspace_bytes")
        ds = _f32(dscore)
        args = (parts.data_ptr(), row_sum.data_ptr(), _ptr(act_mask), ds.data_ptr(), C.byref(g))
        if presorted_ws is not None and tables and c.p.n_branch == 1 and presorted_ws.numel() >= ws_bytes:
            c.launch("nais_pairs_backward_presorted", *args, ws_bytes=ws_bytes, ws=presorted_ws)
        else:
            c.launch("nais_pairs_backward", *args, ws_bytes=ws_bytes)
    return G


def pairs_score(variant: str, beta: float, params: Sequence[torch.Tensor], hist, tgt, hreg=None, treg=None, aux=None,
                dropout_p: float = 0.0, dropout_seed: int = 0, pairs_precision: str = "auto"):
    """Pre-sigmoid scores [B] of explicit pairs (differentiable w.r.t. `params`, ordered as VARIANT_PARAMS[variant]).
    `dropout_p > 0` applies the train-mode dropout of NAIS_basic / NAIS_regionEmbedding (model.py:71,162) with the
    counter-based mask of NaisParams::dropout_seed; backward regenerates the same mask.  `pairs_precision`: "auto" = the
    tcgen05 forward / backward kernels where the shape has them (else the FP32 kernels), "fp32", "tc"."""
    return _PairsFunction.apply(variant, beta, (float(dropout_p), int(dropout_seed), pairs_precision, torch.is_grad_enabled()), hist, tgt, hreg, treg, aux,
                                *params)


def touched_rows(hist, tgt, hreg=None, treg=None) -> Dict[str, torch.Tensor]:
    """Sorted distinct row ids a pair batch touches in each embedding table (int64) — the rows whose gradient is non-zero."""
    if isinstance(hist, SegmentedPairs):
        hist, tgt, hreg, treg = hist.hist, hist.tgt, hist.hreg, hist.treg
    out = {"embed_history.weight": torch.unique(hist), "embed_target.weight": torch.unique(tgt)}
    if hreg is not None:
        out["embed_region.weight"] = torch.unique(torch.cat([hreg.reshape(-1), treg.reshape(-1)]))
    return out


def pairs_backward_compact(variant: str, beta: float, P: Dict[str, torch.Tensor], hist, tgt, hreg, treg, aux, row_sum, parts, dscore,
                           remaps: Dict[str, torch.Tensor], drop=(0.0, 0, "auto"), act_mask: Optional[torch.Tensor] = None):
    """Backward with ROW-COMPACTED table gradients (NaisGrads::remap_*): for every embedding table returns (ids int64 [n] sorted,
    rows float32 [n, w]) of the touched rows only — nothing of size [item_num, w] is allocated, zero-filled or written — plus the
    dense gradients of the remaining (MLP / dist layer) parameters.  `remaps[name]`: a reusable int32 [table rows] scratch per
    table (only the touched entries are rewritten per call).  One-branch variants."""
    dev = _need_cuda(hist, tgt, dscore, *P.values())
    with _PairCall(dev, variant, beta, P, _fwd_bwd(drop[2])[1], drop, (hist, tgt, hreg, treg, aux)) as c:
        if c.p.n_branch != 1:
            raise RuntimeError("row-compacted gradients: one-branch variants only")
        ids = touched_rows(hist, tgt, hreg, treg)
        G = _grad_buffers(P, int(c.b.B), tables=False)
        addr, remap_addr, sparse = _addresses(G), {}, {}
        for name in _TABLES:
            if name not in P or name not in ids:
                continue
            i_ = ids[name]
            rm = remaps[name]
            rm[i_] = torch.arange(i_.numel(), device=dev, dtype=torch.int32)
            rows = torch.empty(i_.numel(), P[name].shape[1], device=dev, dtype=torch.float32)
            addr[name], remap_addr[name] = rows.data_ptr(), rm.data_ptr()
            sparse[name] = (i_, rows)
        g = _grads_struct(variant, addr, remap_addr)
        ds = _f32(dscore)
        c.launch("nais_pairs_backward", parts.data_ptr(), row_sum.data_ptr(), _ptr(act_mask), ds.data_ptr(), C.byref(g),
                 ws_bytes=c.query("nais_pairs_backward_workspace_bytes"))
    return G, sparse


def rows_adagrad(keys: torch.Tensor, rows: torch.Tensor, param: torch.Tensor, state_sum: torch.Tensor, lr: float, eps: float) -> None:
    """nais_rows_adagrad: one row-sparse Adagrad step on `param` / `state_sum` (in place) from key-ordered (id, gradient row) pairs;
    equal ids are summed first, in list order (deterministic).  Ids outside [0, param rows) are skipped."""
    n, w = rows.shape
    if keys.dim() != 1 or keys.shape[0] != n:
        raise RuntimeError(f"rows_adagrad: keys must be 1-D with one id per row ({n}); got {tuple(keys.shape)}")
    if param.dim() != 2 or param.shape[1] != w or state_sum.shape != param.shape:
        raise RuntimeError(f"rows_adagrad: param and its state must be [rows, {w}]; got {tuple(param.shape)} and {tuple(state_sum.shape)}")
    dev = _need_cuda(keys, rows, param, state_sum)
    lib = _lib.load()
    if not (param.is_contiguous() and state_sum.is_contiguous() and param.dtype == torch.float32 and state_sum.dtype == torch.float32):
        raise RuntimeError("rows_adagrad: param and its state must be contiguous float32")
    with torch.cuda.device(dev):
        # (clamped before the int32 cast: an id >= 2**31 or >= 2**32 stays out of range instead of wrapping onto a real row; the
        # clamp is monotone, so the list stays in key order)
        k32 = keys.clamp(-1, param.shape[0]).to(torch.int32).contiguous()
        r = _f32(rows)
        ws_bytes = lib.nais_rows_adagrad_workspace_bytes(n, w)
        ws = torch.empty(max(ws_bytes, 16), device=dev, dtype=torch.uint8)
        _lib.check(lib.nais_rows_adagrad(k32.data_ptr(), r.data_ptr(), n, w, param.shape[0], None, param.data_ptr(), state_sum.data_ptr(),
                                         float(lr), float(eps), ws.data_ptr(), ws_bytes, _stream()), "nais_rows_adagrad")


def pairs_backward_adagrad(variant: str, beta: float, P: Dict[str, torch.Tensor], sums: Dict[str, torch.Tensor], lr: float,
                           eps: float, hist, tgt, hreg, treg, aux, row_sum, parts, dscore, drop=(0.0, 0, "auto"),
                           act_mask: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Backward of `pairs_score` with the embedding tables stepped in place by a row-sparse Adagrad fused into the
    sorted-segment reduce (nais_pairs_backward_adagrad; replaces run.py:252-254 for `embed_*`): `sums[name]` is the
    optimizer's `state['sum']` of table `name`; P[name] and sums[name] of every touched row are updated, nothing dense is
    written.  Returns the gradients of the remaining (MLP / dist layer / embed_distance) parameters."""
    dev = _need_cuda(hist, tgt, dscore, *P.values())
    with _PairCall(dev, variant, beta, P, _fwd_bwd(drop[2])[1], drop, (hist, tgt, hreg, treg, aux)) as c:
        G = _grad_buffers(P, int(c.b.B), tables=False)
        g = _grads_struct(variant, _addresses(G))
        o = _adagrad_struct(variant, P, sums, lr, eps, tables=True)
        ds = _f32(dscore)
        c.launch("nais_pairs_backward_adagrad", parts.data_ptr(), row_sum.data_ptr(), _ptr(act_mask), ds.data_ptr(), C.byref(g),
                 C.byref(o), ws_bytes=c.query("nais_pairs_backward_workspace_bytes"))
    return G


def pairs_train_step(variant: str, beta: float, P: Dict[str, torch.Tensor], table_sums: Dict[str, torch.Tensor],
                     dense_sums: Dict[str, torch.Tensor], lr_tables: float, eps_tables: float, lr_dense: float, eps_dense: float,
                     label: torch.Tensor, hist, tgt=None, hreg=None, treg=None, aux=None, row_weight: Optional[torch.Tensor] = None,
                     drop=(0.0, 0, "auto"), want_score: bool = False):
    """nais_pairs_train_step: zero_grad -> forward -> sigmoid + BCELoss -> backward -> Adagrad.step of run.py:248-254 in ONE
    library call (8-12 launches).  Every tensor of `P` and every `state['sum']` in `table_sums` / `dense_sums` is updated in
    place.  Returns (loss [1] on the device, pre-sigmoid scores [B] or None)."""
    dev = _need_cuda(hist, tgt, label, *P.values())
    with _PairCall(dev, variant, beta, P, drop[2], drop, (hist, tgt, hreg, treg, aux)) as c:
        o = _adagrad_struct(variant, P, table_sums, lr_tables, eps_tables, tables=True)
        d = _adagrad_struct(variant, P, dense_sums, lr_dense, eps_dense, tables=False)
        lab = _f32(label)
        rw = None if row_weight is None else _f32(row_weight)
        ws_bytes = c.query("nais_pairs_train_step_workspace_bytes")
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        score = torch.empty(int(c.b.B), device=dev, dtype=torch.float32) if want_score else None
        c.launch("nais_pairs_train_step", lab.data_ptr(), _ptr(rw), C.byref(o), C.byref(d), loss.data_ptr(), _ptr(score),
                 ws_bytes=ws_bytes)
    return loss, score


def pairs_train_step_bpr(variant: str, beta: float, P: Dict[str, torch.Tensor], table_sums: Dict[str, torch.Tensor],
                         dense_sums: Dict[str, torch.Tensor], lr_tables: float, eps_tables: float, lr_dense: float, eps_dense: float,
                         num_neg: int, hist, tgt=None, hreg=None, treg=None, aux=None, group_weight: Optional[torch.Tensor] = None,
                         drop=(0.0, 0, "auto"), want_score: bool = False):
    """nais_pairs_train_step_bpr: `pairs_train_step` with the BPR loss -log sigmoid(s+ - s-) in ONE library call.  The rows come in
    groups of 1 + num_neg (positive first: the order of DeviceBatcher.batch / multi_user_batch); the loss is the mean over the
    (positive, negative) pairs, or sum_g group_weight[g] * sum_j softplus(s_g,j - s_g,0) with `group_weight` [n_groups].  Updates
    `P` and the optimizer sums in place.  Returns (loss [1] on the device, pre-sigmoid scores [B] or None)."""
    dev = _need_cuda(hist, tgt, group_weight, *P.values())
    with _PairCall(dev, variant, beta, P, drop[2], drop, (hist, tgt, hreg, treg, aux)) as c:
        o = _adagrad_struct(variant, P, table_sums, lr_tables, eps_tables, tables=True)
        d = _adagrad_struct(variant, P, dense_sums, lr_dense, eps_dense, tables=False)
        gw = None if group_weight is None else _f32(group_weight)
        if gw is not None and gw.numel() * (num_neg + 1) != int(c.b.B):
            raise RuntimeError(f"pairs_train_step_bpr: one group weight per group of {num_neg + 1} rows")
        bpr = _lib.NaisBprLoss(int(num_neg), 0, _ptr(gw))
        ws_bytes = c.query("nais_pairs_train_step_workspace_bytes")
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        score = torch.empty(int(c.b.B), device=dev, dtype=torch.float32) if want_score else None
        c.launch("nais_pairs_train_step_bpr", C.byref(bpr), C.byref(o), C.byref(d), loss.data_ptr(), _ptr(score), ws_bytes=ws_bytes)
    return loss, score


def train_users(variant: str, beta: float, P: Dict[str, torch.Tensor], table_sums, dense_sums, lr_tables, eps_tables, lr_dense,
                eps_dense, host_indptr, indices: torch.Tensor, entry_region: Optional[torch.Tensor],
                entry_coords: Optional[torch.Tensor], poi_region: Optional[torch.Tensor], poi_coords: Optional[torch.Tensor],
                users, num_ng: int, seed: int, pairs_precision: str = "auto", center: Tuple[float, float] = (0.0, 0.0),
                dropout_p: float = 0.0, dropout_seeds=None, loss: str = "bce") -> torch.Tensor:
    """nais_train_users: the reference's schedule, one optimizer step per user (run.py:227-255), for a list of users in ONE library
    call — per user the device sampler over his CSR slice + the one-call training step, ~15 launches and no host work in between.
    `host_indptr` / `users`: numpy int64 (host).  `center`: the (lat, lon) subtracted from `entry_coords` / `poi_coords`.
    `dropout_p > 0`: train-mode dropout, the step of users[i] with mask seed `dropout_seeds[i]` (host, one per user; entries of
    users without a history are ignored).  `loss`: "bce" (the reference's batch-mean BCE) or "bpr" (nais_train_users_bpr: the mean
    BPR loss over the user's positive / negative pairs).  Updates every tensor of `P` and the optimizer sums in place; returns the
    per-user losses [n] (device)."""
    import numpy as np
    entry = {"bce": "nais_train_users_dropout", "bpr": "nais_train_users_bpr"}.get(loss)
    if entry is None:
        raise ValueError(f"train_users: loss must be 'bce' or 'bpr', not {loss!r}")
    dev = _need_cuda(indices, entry_region, entry_coords, poi_region, poi_coords, *P.values())
    hp = np.ascontiguousarray(np.asarray(host_indptr, dtype=np.int64))
    hu = np.ascontiguousarray(np.asarray(users, dtype=np.int64))
    if hu.size and (hu.min() < 0 or hu.max() + 1 >= hp.size):
        raise IndexError("train_users: user id outside the train matrix")
    ds = None
    if dropout_p > 0:
        ds = np.ascontiguousarray(np.asarray(dropout_seeds, dtype=np.uint64).reshape(-1))
        if ds.size != hu.size:
            raise RuntimeError("train_users: one dropout seed per user")
    with _PairCall(dev, variant, beta, P, pairs_precision, (float(dropout_p), 0)) as c:
        o = _adagrad_struct(variant, P, table_sums, lr_tables, eps_tables, tables=True)
        d = _adagrad_struct(variant, P, dense_sums, lr_dense, eps_dense, tables=False)
        if indices.dtype != torch.int64 or not indices.is_contiguous():
            raise RuntimeError("train_users: `indices` must be contiguous int64 (the CSR of the train matrix)")
        er = None if entry_region is None else entry_region.to(torch.int64).contiguous()
        ec = None if entry_coords is None else _f32(entry_coords)
        pr = None if poi_region is None else poi_region.to(torch.int32).contiguous()
        pc = None if poi_coords is None else _f32(poi_coords)
        max_hist = int((hp[hu + 1] - hp[hu]).max()) if hu.size else 0
        losses = torch.empty(max(hu.size, 1), device=dev, dtype=torch.float32)
        c.launch(entry, hp.ctypes.data, int(hp.size) - 1, indices.data_ptr(), _ptr(er), _ptr(ec), _ptr(pr), _ptr(pc),
                 hu.ctypes.data, int(hu.size), int(num_ng), int(seed) & (2 ** 64 - 1), C.byref(o), C.byref(d), losses.data_ptr(),
                 ws_bytes=c.query("nais_train_users_workspace_bytes", max(max_hist, 1), int(num_ng)),
                 tail=(float(center[0]), float(center[1]), None if ds is None else ds.ctypes.data))
    return losses[: hu.size]


def pairs_forward_raw(variant: str, beta: float, P: Dict[str, torch.Tensor], hist, tgt, hreg, treg, aux, drop=(0.0, 0, "auto")):
    """(score[B], row_sum, parts, act_mask) of nais_pairs_forward without autograd bookkeeping (the fused train step keeps
    them for its backward; act_mask is None unless the tcgen05 forward ran)."""
    dev = _need_cuda(hist, tgt, *P.values())
    with _PairCall(dev, variant, beta, P, _fwd_bwd(drop[2])[0], drop, (hist, tgt, hreg, treg, aux)) as c:
        score, row_sum, parts, mask, _ = _forward_launch(c)
    return score, row_sum, parts, mask


def pairs_explain(variant: str, beta: float, P: Dict[str, torch.Tensor], hist, tgt=None, hreg=None, treg=None, aux=None, m: int = 5,
                  precision: str = "auto"):
    """Why each pair scored what it did (nais_pairs_explain): (score [B] pre-sigmoid, bit-identical to the pair forward's; pos
    [B,m] int64, the m history positions with the largest contribution c_h = sum_b E_bh s_bh / S_b^beta, descending, ties by
    ascending position; contrib [B,m] those c_h (summed over all h they are the score); attn [n_branch,B,m] their attention
    share E_bh / S_b).  Masked positions (history item == target) are never selected; rows with fewer than m selectable positions
    are padded with pos -1, contrib -inf, attn 0.  `pos` indexes the row's own history: hist[b, pos], or for an ops.SegmentedPairs
    `hist` the segment's slice of hist.hist.  `precision`: the pair forward's kernels ("auto", "fp32", "tc").  No dropout, no
    autograd."""
    dev = _need_cuda(hist, tgt, hreg, treg, aux, *P.values())
    m = int(m)
    if not 1 <= m <= 32:
        raise ValueError(f"pairs_explain: m must be in [1, 32], got {m}")
    with _PairCall(dev, variant, beta, P, precision, batch=(hist, tgt, hreg, treg, aux)) as c:
        B, nb = int(c.b.B), int(c.p.n_branch)
        score = torch.empty(B, device=dev, dtype=torch.float32)
        pos = torch.empty(B, m, device=dev, dtype=torch.int32)
        contrib = torch.empty(B, m, device=dev, dtype=torch.float32)
        attn = torch.empty(nb, B, m, device=dev, dtype=torch.float32)
        c.launch("nais_pairs_explain", m, score.data_ptr(), pos.data_ptr(), contrib.data_ptr(), attn.data_ptr(),
                 ws_bytes=c.query("nais_pairs_explain_workspace_bytes"))
    return score, pos.to(torch.int64), contrib, attn


def dropout_keep_mask(seed: int, B: int, H: int, hid: int, p: float):
    """The keep-mask the kernels use for a dense [B,H] batch, on the host (numpy bool [B,H,hid]) — for tests / reproducing a step."""
    return dropout_keep_mask_cells(seed, B * H, hid, p).reshape(B, H, hid)


def dropout_keep_mask_cells(seed: int, n_cells: int, hid: int, p: float):
    """The keep-mask of `n_cells` cells on the host (numpy bool [n_cells, hid]), indexed by the per-cell index of NaisPairs: b*H + h
    for a dense batch, seg_cell_offsets[s] + (r - row_offsets[s]) * H_s + h for a segmented one (include/nais_b200.h)."""
    import numpy as np
    idx = np.arange(n_cells * hid, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    t = min(int(float(np.float32(p)) * 4294967296.0), 0xFFFFFFFF)
    return ((z >> np.uint64(32)) >= np.uint64(t)).reshape(n_cells, hid)


# ----------------------------------------------------------------------------------------------------------------------
# Full-rank scoring + top-k
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class DeviceCatalog:
    """Candidate-side arrays resident on the device (replaces businessRegionEmbedList + latlon_mat arguments of
    validation.py:62).  coords are centred in float64 on the host before the float32 cast (DESIGN.md §precision)."""
    region: Optional[torch.Tensor]  # [n_rows] int32
    coords: Optional[torch.Tensor]  # [n_rows,2] float32, centred
    row_base: int
    n_rows: int
    center: Tuple[float, float]


@dataclass
class DeviceUsers:
    offsets: torch.Tensor  # [U+1] int64 (device)
    items: torch.Tensor  # [nnz] int32
    region: Optional[torch.Tensor]  # [nnz] int32
    coords: Optional[torch.Tensor]  # [nnz,2] float32 centred
    n_users: int
    nnz: int
    host_offsets: Optional[object] = None  # numpy copy of `offsets` (lets predict_topk split huge batches by workspace size)

    def slice(self, u0: int, u1: int) -> "DeviceUsers":
        """Users [u0, u1) as a new DeviceUsers (offsets rebased); needs `host_offsets`."""
        ho = self.host_offsets
        a, b = int(ho[u0]), int(ho[u1])
        return DeviceUsers((self.offsets[u0:u1 + 1] - a).contiguous(), self.items[a:b], None if self.region is None else self.region[a:b],
                           None if self.coords is None else self.coords[a:b], u1 - u0, b - a, ho[u0:u1 + 1] - a)


def _structs(cat: DeviceCatalog, users: Optional[DeviceUsers]):
    c = NaisCatalog()
    c.region, c.coords, c.row_base, c.n_rows = _ptr(cat.region), _ptr(cat.coords), cat.row_base, cat.n_rows
    c.center_lat, c.center_lon = float(cat.center[0]), float(cat.center[1])
    if users is None:
        return c, None
    u = NaisUsers()
    u.offsets, u.items, u.region, u.coords, u.n_users = (_ptr(users.offsets), _ptr(users.items), _ptr(users.region),
                                                         _ptr(users.coords), users.n_users)
    return c, u


WORKSPACE_LIMIT_BYTES = 8 << 30  # user batches whose workspace would exceed this are scored in slices


def _tensor_path_device(dev: torch.device) -> bool:
    return torch.cuda.get_device_capability(dev)[0] == 10  # tcgen05 / TMEM: sm_100 family only


def resolve_precision(lib, p, precision: str, dev: Optional[torch.device] = None) -> str:
    """"auto" = the tensor-core path with its device-side MIX/SPLIT gate ("tc_auto") wherever the model shape has one
    (every variant of model.py incl. the two-branch disentangled one; D and hid up to 256 in steps of 16/32 — csrc/nais_tc.cu make_geo) and the device is sm_100,
    else the FP32 kernel."""
    if precision != "auto":
        return precision
    if dev is not None and not _tensor_path_device(dev):
        return "fp32"
    return "tc_auto" if lib.nais_fullrank_workspace_bytes(C.byref(p), 1, 1, 0, min(128, p.item_num), 1, PRECISIONS["tc_auto"]) else "fp32"


@dataclass
class FullrankPlan:
    """Everything `nais_fullrank_topk` would recompute per call although it depends only on the weights and the catalogue
    range (table maxima, scales, hidden-unit permutation, packed candidate image; include/nais_b200.h
    `nais_fullrank_prepare`).  Valid until a parameter, the catalogue or the range changes."""
    buf: Optional[torch.Tensor]  # device bytes (None: FP32 precision needs no plan)
    precision: str
    poi_begin: int
    poi_end: int
    key: tuple = ()

    @property
    def nbytes(self) -> int:
        return 0 if self.buf is None else self.buf.numel()

    def tc_choice(self) -> Optional[Dict[str, float]]:
        """What the device-side gate of this plan decided: `rho` (bound on the logit scale) and `use_mix` (1 = the fp16 +
        e5m2-correction kernels score every user with at least `min_hist_for_mix` history items under "tc_auto", 0 = the
        three-pass fp16 split scores everyone).  Synchronises."""
        if self.buf is None:
            return None
        host = self.buf[64:128].cpu()
        return {"rho": float(host[44:48].view(torch.float32).item()), "use_mix": int(host[48:52].view(torch.int32).item()),
                "min_hist_for_mix": 16, "rho_max_for_mix": 128.0}  # kMixRhoMax / kMixMinHist in csrc/nais_tc.cu


def fullrank_prepare(variant: str, beta: float, P: Dict[str, torch.Tensor], cat: "DeviceCatalog", poi_begin: int = 0,
                     poi_end: Optional[int] = None, precision: str = "auto") -> FullrankPlan:
    """Build the plan of (weights, catalogue range, precision): once per evaluation, not once per user batch."""
    dev = _need_cuda(cat.region, cat.coords, *P.values())
    lib = _lib.load()
    keep: List[torch.Tensor] = []
    with torch.cuda.device(dev):
        p = build_params(variant, P, beta, keep)
        poi_end = p.item_num if poi_end is None else poi_end
        precision = resolve_precision(lib, p, precision, dev)
        prec = PRECISIONS[precision]
        nbytes = lib.nais_fullrank_plan_bytes(C.byref(p), poi_begin, poi_end, prec)
        if precision == "fp32" or poi_end <= poi_begin:
            return FullrankPlan(None, precision, poi_begin, poi_end)
        if nbytes == 0:
            raise RuntimeError(f"precision {precision!r} has no tensor path for this model shape")
        buf = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        c, _ = _structs(cat, None)
        _lib.check(lib.nais_fullrank_prepare(C.byref(p), C.byref(c), poi_begin, poi_end, prec, buf.data_ptr(), nbytes, _stream()),
                   "nais_fullrank_prepare")
    _LAST_TC_PLAN[0] = FullrankPlan(buf, precision, poi_begin, poi_end)
    return _LAST_TC_PLAN[0]


@dataclass
class GeoMix:
    """Power-law geo re-ranking of a full-rank call (include/nais_b200.h NaisGeoMix): rank by
    (1 - alpha) * sigmoid(score) + alpha * exp(log G - M_u), log G = sum_h ln(a * max(0.01, d_km)^b).  `logmax` [U] float32 on
    the device holds M_u over the whole ranked catalogue (`powerlaw_logmax`, max-combined across shards)."""
    a: float
    b: float
    alpha: float
    logmax: torch.Tensor

    def slice(self, u0: int, u1: int) -> "GeoMix":
        return GeoMix(self.a, self.b, self.alpha, self.logmax[u0:u1])


def powerlaw_logmax(cat: DeviceCatalog, users: DeviceUsers, a: float, b: float, poi_begin: int = 0, poi_end: Optional[int] = None,
                    exclude_history: bool = True) -> torch.Tensor:
    """M_u = max_j log G(u, j) over [poi_begin, poi_end) (minus the history when `exclude_history`) [U] float32, -inf for a user
    without candidates (nais_powerlaw_logmax; bit-identical to the maximum of powerlaw.log_scores, no [U, N] buffer)."""
    dev = _need_cuda(users.offsets, cat.coords)
    lib = _lib.load()
    poi_end = cat.row_base + cat.n_rows if poi_end is None else poi_end
    out = torch.empty(users.n_users, device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        c, u = _structs(cat, users)
        _lib.check(lib.nais_powerlaw_logmax(C.byref(c), C.byref(u), poi_begin, poi_end, float(a), float(b), int(exclude_history),
                                            out.data_ptr(), _stream()), "nais_powerlaw_logmax")
    return out


def fullrank_topk(variant: str, beta: float, P: Dict[str, torch.Tensor], cat: DeviceCatalog, users: DeviceUsers, k: int,
                  poi_begin: int = 0, poi_end: Optional[int] = None, exclude_history: bool = True,
                  precision: str = "fp32", plan: Optional[FullrankPlan] = None, return_keys: bool = False,
                  geo: Optional[GeoMix] = None):
    """(score[U,k] pre-sigmoid descending, id[U,k] int32 global POI ids; -inf / -1 padding) — or, with `return_keys`, the
    packed ranking keys [U,k] int64 (bit pattern of the uint64 keys `topk_merge_keys` consumes).  `plan`: a
    `fullrank_prepare` result for the same weights / range / precision; without one the constants are recomputed by this
    call (`nais_fullrank_topk`).  `geo`: rank by the power-law mix instead (`nais_fullrank_topk_geo_planned`, always planned);
    the score is then the mixed value, not a pre-sigmoid score."""
    dev = _need_cuda(users.offsets, users.items, users.region, users.coords, cat.region, cat.coords, *P.values())
    lib = _lib.load()
    keep: List[torch.Tensor] = []
    with torch.cuda.device(dev):
        p = build_params(variant, P, beta, keep)
        poi_end = p.item_num if poi_end is None else poi_end
        if plan is not None:
            if (plan.poi_begin, plan.poi_end) != (poi_begin, poi_end):
                raise RuntimeError("the plan was prepared for another catalogue range")
            precision = plan.precision
        precision = resolve_precision(lib, p, precision, dev)
        prec = PRECISIONS[precision]
        planned = plan is not None or return_keys or geo is not None
        if planned:
            ws_bytes = lib.nais_fullrank_planned_workspace_bytes(C.byref(p), users.n_users, users.nnz, poi_begin, poi_end, k, prec)
        else:
            ws_bytes = lib.nais_fullrank_workspace_bytes(C.byref(p), users.n_users, users.nnz, poi_begin, poi_end, k, prec)
        if ws_bytes > WORKSPACE_LIMIT_BYTES and users.host_offsets is not None and users.n_users > 1:
            n_slices = min(users.n_users, -(-ws_bytes // WORKSPACE_LIMIT_BYTES))
            step = -(-users.n_users // n_slices)
            parts = [fullrank_topk(variant, beta, P, cat, users.slice(u0, min(users.n_users, u0 + step)), k, poi_begin, poi_end,
                                   exclude_history, precision, plan, return_keys,
                                   None if geo is None else geo.slice(u0, min(users.n_users, u0 + step)))
                     for u0 in range(0, users.n_users, step)]
            if return_keys:
                return torch.cat(parts)
            return torch.cat([a for a, _ in parts]), torch.cat([b for _, b in parts])
        if planned and plan is None:
            plan = fullrank_prepare(variant, beta, P, cat, poi_begin, poi_end, precision)
        c, u = _structs(cat, users)
        ws = torch.empty(max(ws_bytes, 16), device=dev, dtype=torch.uint8)
        if return_keys:
            out_k = torch.empty(users.n_users, k, device=dev, dtype=torch.int64)
            out_s = out_i = None
        else:
            out_k = None
            out_s = torch.empty(users.n_users, k, device=dev, dtype=torch.float32)
            out_i = torch.empty(users.n_users, k, device=dev, dtype=torch.int32)
        if geo is not None:
            if geo.logmax.numel() != users.n_users or geo.logmax.device != dev or geo.logmax.dtype != torch.float32:
                raise ValueError("geo.logmax must be a float32 [n_users] tensor on the users' device")
            lm = geo.logmax.contiguous()
            g = _lib.NaisGeoMix(float(geo.a), float(geo.b), float(geo.alpha), lm.data_ptr())
            _lib.check(lib.nais_fullrank_topk_geo_planned(C.byref(p), C.byref(c), C.byref(u), poi_begin, poi_end, k,
                                                          int(exclude_history), prec, _ptr(plan.buf), plan.nbytes, C.byref(g),
                                                          _ptr(out_k), _ptr(out_s), _ptr(out_i), ws.data_ptr(), ws_bytes, _stream()),
                       "nais_fullrank_topk_geo_planned")
        elif planned:
            _lib.check(lib.nais_fullrank_topk_planned(C.byref(p), C.byref(c), C.byref(u), poi_begin, poi_end, k, int(exclude_history),
                                                      prec, _ptr(plan.buf), plan.nbytes, _ptr(out_k), _ptr(out_s), _ptr(out_i),
                                                      ws.data_ptr(), ws_bytes, _stream()), "nais_fullrank_topk_planned")
        else:
            _lib.check(lib.nais_fullrank_topk(C.byref(p), C.byref(c), C.byref(u), poi_begin, poi_end, k, int(exclude_history),
                                              prec, out_s.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws_bytes, _stream()),
                       "nais_fullrank_topk")
            if precision != "fp32" and ws_bytes >= 128 and users.n_users and poi_end > poi_begin:
                # device-side scales / precision gate of this call (the plan sits at the head of the workspace), read lazily by
                # last_tc_choice(); a 128-byte copy, not a view: a view would pin the whole (up to 8 GiB) workspace
                _LAST_TC_PLAN[0] = FullrankPlan(ws[:128].clone(), precision, poi_begin, poi_end)
    return out_k if return_keys else (out_s, out_i)


_LAST_TC_PLAN: List[Optional[FullrankPlan]] = [None]


def last_tc_choice() -> Optional[Dict[str, float]]:
    """`FullrankPlan.tc_choice()` of the last tensor-path plan built or call made.  Synchronises."""
    return None if _LAST_TC_PLAN[0] is None else _LAST_TC_PLAN[0].tc_choice()


def topk_merge_keys(keys: torch.Tensor, want_keys: bool = False):
    """Merge key lists [L, U, k] (int64 bit patterns of the uint64 ranking keys; L = one list per catalogue shard, exactly
    the layout `all_gather_into_tensor` produces) into (score [U,k], id [U,k] int32) — or the merged keys [U,k]."""
    dev = _need_cuda(keys)
    L, U, k = keys.shape
    lib = _lib.load()
    with torch.cuda.device(dev):
        kk = keys.contiguous()
        if want_keys:
            out_k = torch.empty(U, k, device=dev, dtype=torch.int64)
            out_s = out_i = None
        else:
            out_k = None
            out_s = torch.empty(U, k, device=dev, dtype=torch.float32)
            out_i = torch.empty(U, k, device=dev, dtype=torch.int32)
        _lib.check(lib.nais_topk_merge_keys(kk.data_ptr(), k, U * k, U, L, k, _ptr(out_k), _ptr(out_s), _ptr(out_i), _stream()),
                   "nais_topk_merge_keys")
    return out_k if want_keys else (out_s, out_i)


def keys_to_lists(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Unpack ranking keys (ordered(score) << 32 | (0xFFFFFFFF - id), 0 = no entry; csrc/nais_common.cuh make_key) into
    (score float32, id int32; -inf / -1 padding).  Bit arithmetic on the int64 bit patterns: works on any device (the gloo
    CPU tests of the sharding logic use it); the CUDA path never needs it — nais_topk_merge_keys writes score / id itself."""
    o = (keys >> 32) & 0xFFFFFFFF
    bits = torch.where((o & 0x80000000) != 0, o & 0x7FFFFFFF, (~o) & 0xFFFFFFFF)
    score = torch.where(bits >= 2 ** 31, bits - 2 ** 32, bits).to(torch.int32).view(torch.float32).clone()
    ids = (0xFFFFFFFF - (keys & 0xFFFFFFFF)).to(torch.int32)
    empty = keys == 0
    score[empty] = float("-inf")
    ids[empty] = -1
    return score, ids


def lists_to_keys(score: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    """Inverse of `keys_to_lists` (same packing as make_key: NaN ranks as -inf, id < 0 = no entry -> key 0)."""
    sc = torch.where(torch.isnan(score), torch.full_like(score, float("-inf")), score).to(torch.float32).contiguous()
    u = sc.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    o = torch.where((u & 0x80000000) != 0, (~u) & 0xFFFFFFFF, u | 0x80000000)
    lo = 0xFFFFFFFF - ids.to(torch.int64)
    hi = torch.where(o >= 2 ** 31, o - 2 ** 32, o)  # the top half as a signed 32-bit value, so the shift stays inside int64
    keys = (hi << 32) | lo
    return torch.where(ids < 0, torch.zeros_like(keys), keys)


def fullrank_scores(variant: str, beta: float, P: Dict[str, torch.Tensor], cat: DeviceCatalog, users: DeviceUsers,
                    poi_begin: int = 0, poi_end: Optional[int] = None, precision: str = "fp32") -> torch.Tensor:
    """All pre-sigmoid scores [U, poi_end-poi_begin] through the fused path (small cases / parity checks)."""
    dev = _need_cuda(users.offsets, users.items, users.region, users.coords, cat.region, cat.coords, *P.values())
    lib = _lib.load()
    keep: List[torch.Tensor] = []
    with torch.cuda.device(dev):
        p = build_params(variant, P, beta, keep)
        poi_end = p.item_num if poi_end is None else poi_end
        c, u = _structs(cat, users)
        precision = resolve_precision(lib, p, precision, dev)
        prec = PRECISIONS[precision]
        out = torch.empty(users.n_users, poi_end - poi_begin, device=dev, dtype=torch.float32)
        ws_bytes = lib.nais_fullrank_workspace_bytes(C.byref(p), users.n_users, users.nnz, poi_begin, poi_end, 1, prec)
        ws = torch.empty(max(ws_bytes, 16), device=dev, dtype=torch.uint8)
        _lib.check(lib.nais_fullrank_scores(C.byref(p), C.byref(c), C.byref(u), poi_begin, poi_end, prec, out.data_ptr(),
                                            ws.data_ptr(), ws_bytes, _stream()), "nais_fullrank_scores")
    return out


def topk_merge(scores: torch.Tensor, ids: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Merge [U, L, k] lists (one per catalogue shard) into [U, k] by (score desc, id asc)."""
    dev = _need_cuda(scores, ids)
    U, L, k = scores.shape
    lib = _lib.load()
    with torch.cuda.device(dev):
        s, i = _f32(scores), ids.to(torch.int32).contiguous()
        out_s = torch.empty(U, k, device=dev, dtype=torch.float32)
        out_i = torch.empty(U, k, device=dev, dtype=torch.int32)
        _lib.check(lib.nais_topk_merge(s.data_ptr(), i.data_ptr(), U, L, k, out_s.data_ptr(), out_i.data_ptr(), _stream()),
                   "nais_topk_merge")
    return out_s, out_i


def hits_at_k(rec_ids: torch.Tensor, positives: Sequence[Sequence[int]], k_list: Sequence[int]) -> torch.Tensor:
    """hits[U, len(k_list)] = |set(positives[u]) & set(rec_ids[u, :k])| on the device (nais_hits_at_k) — the integer core
    of eval_metrics.precision_at_k / recall_at_k / hitrate_at_k (eval_metrics.py:36-69)."""
    import numpy as np
    dev = _need_cuda(rec_ids)
    U, k_rec = rec_ids.shape
    lens = np.fromiter((len(p) for p in positives), dtype=np.int64, count=U)
    off = np.zeros(U + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    flat = np.fromiter((int(x) for p in positives for x in p), dtype=np.int32, count=int(off[-1]))
    lib = _lib.load()
    with torch.cuda.device(dev):
        rec = rec_ids.to(torch.int32).contiguous()
        po = torch.from_numpy(off).to(dev)
        pi = torch.from_numpy(flat).to(dev) if len(flat) else torch.zeros(1, dtype=torch.int32, device=dev)
        kl = torch.tensor(list(k_list), dtype=torch.int32, device=dev)
        hits = torch.empty(U, len(k_list), dtype=torch.int32, device=dev)
        _lib.check(lib.nais_hits_at_k(rec.data_ptr(), U, k_rec, po.data_ptr(), pi.data_ptr(), kl.data_ptr(), len(k_list),
                                      hits.data_ptr(), _stream()), "nais_hits_at_k")
    return hits
