"""Drop-in for the NAIS batch builders of the reference's `batches.py` (:67-139).

Same arguments, same outputs (int64 / float32 tensors on the CUDA device), same use of Python's global `random`
stream — so `random.seed(s)` gives the batch the reference would build — but the O(N) Python `set` difference is a
numpy mask.
"""
from __future__ import annotations

import random

import numpy as np
import torch


def _device():
    return torch.device("cuda" if torch.cuda.is_available() else "cpu")


def _non_visited(num_poi: int, visited) -> list:
    m = np.ones(num_poi, dtype=bool)
    m[np.asarray(visited, dtype=np.int64)] = False
    return np.nonzero(m)[0].tolist()  # ascending == CPython iteration order of set(range(N)) - set(visited)


def get_NAIS_batch_region(train_matrix, num_poi, uid, negative_num, businessRegionEmbedList):
    """Per-user training batch (batches.py:67-108): shuffled positives, `len(pos)*negative_num` negatives drawn as the
    head of a shuffle of all non-visited POIs, targets interleaved [p, n..n], labels [1, 0..0], history repeated."""
    dev = _device()
    region = np.asarray(businessRegionEmbedList)
    positives = train_matrix.getrow(uid).indices.tolist()
    random.shuffle(positives)
    negative = _non_visited(num_poi, positives)
    random.shuffle(negative)
    negatives = np.array(negative[:len(positives) * negative_num], dtype=np.int64).reshape(-1, negative_num)
    pos = np.array(positives, dtype=np.int64)
    data = np.concatenate((pos.reshape(-1, 1), negatives), axis=-1).reshape(-1)
    labels = np.tile(np.array([1.0] + [0.0] * negative_num, dtype=np.float32), len(positives))
    hist = np.broadcast_to(pos, (len(data), len(pos)))
    return (torch.from_numpy(np.ascontiguousarray(hist)).to(dev), torch.from_numpy(data).to(dev),
            torch.from_numpy(labels).to(dev), torch.from_numpy(np.ascontiguousarray(region[hist]).astype(np.int64)).to(dev),
            torch.from_numpy(region[data].astype(np.int64)).to(dev))


def get_NAIS_batch_test_region(train_matrix, uid, businessRegionEmbedList):
    """Per-user full-catalogue test batch (batches.py:110-139)."""
    dev = _device()
    region = np.asarray(businessRegionEmbedList)
    history = np.asarray(train_matrix.getrow(uid).indices, dtype=np.int64)
    negative = np.asarray(_non_visited(train_matrix.shape[1], history), dtype=np.int64)
    hist = np.broadcast_to(history, (len(negative), len(history)))
    label = torch.zeros(len(negative), dtype=torch.float32, device=dev)
    return (torch.from_numpy(np.ascontiguousarray(hist)).to(dev), torch.from_numpy(negative).to(dev), label,
            torch.from_numpy(np.ascontiguousarray(region[hist]).astype(np.int64)).to(dev),
            torch.from_numpy(region[negative].astype(np.int64)).to(dev))


def get_NAIS_batch(train_matrix, num_poi, uid, negative_num):
    """batches.py:24-50 (no regions)."""
    h, t, l, _, _ = get_NAIS_batch_region(train_matrix, num_poi, uid, negative_num, np.zeros(num_poi, dtype=np.int64))
    return h, t, l


def get_NAIS_batch_test(train_matrix, uid):
    """batches.py:52-65."""
    h, t, l, _, _ = get_NAIS_batch_test_region(train_matrix, uid, np.zeros(train_matrix.shape[1], dtype=np.int64))
    return h, t, l


def lat_lon_pairs(place_coords, target_pois, history_pois, device=None):
    """ll[b,h,:] = |coords[target_b] - coords[history_h]| as float32: the values the reference gathers from its dense
    float64 `latlon_mat` (run.py:47-54,239-247) without building the O(N^2) table."""
    c = np.asarray(place_coords, dtype=np.float64)
    t = np.asarray(target_pois, dtype=np.int64)
    h = np.asarray(history_pois, dtype=np.int64)
    if h.ndim == 1:
        h = np.broadcast_to(h, (len(t), len(h)))
    ll = np.abs(c[t][:, None, :] - c[h]).astype(np.float32)
    return torch.from_numpy(ll).to(device or _device())


def dist_km_pairs(place_coords, target_pois, history_pois, device=None):
    """km[b,h] = great-circle km between target_b and history_h (powerLaw.dist in float64, cast to float32): the `target_distance`
    argument of NAIS_region_distance_disentangled_Embedding (model.py:497-504) for a dense [B,H] batch."""
    from .powerlaw import dist
    c = np.asarray(place_coords, dtype=np.float64)
    t = np.asarray(target_pois, dtype=np.int64)
    h = np.asarray(history_pois, dtype=np.int64)
    if h.ndim == 1:
        h = np.broadcast_to(h, (len(t), len(h)))
    km = dist((c[t][:, None, 0], c[t][:, None, 1]), (c[h][..., 0], c[h][..., 1])).astype(np.float32)
    return torch.from_numpy(np.ascontiguousarray(km)).to(device or _device())


class DeviceBatcher:
    """Training batches built ON THE DEVICE (SURVEY.md §8 f1): same batch layout as `get_NAIS_batch_region`
    (batches.py:67-108: shuffled positives, targets interleaved [p, n..n], labels [1, 0..0], history repeated per target)
    and the same sampling *distribution* — `len(pos)*num_ng` negatives uniform without replacement over the non-visited
    POIs — but drawn with a device RNG (`torch.randperm`), not the reference's Python `random` stream, and without any
    O(N) Python list work or host->device copies per user.  Also returns the |dlat|,|dlon| tensor of run.py:239-247.

    `batch` (one user, dense layout) is PyTorch index plumbing; `multi_user_batch` (many users, segmented layout) samples
    with the library's `nais_sample_batch` kernel and materialises neither the [B,H] history repeat nor the [B,H,2] tensor."""

    def __init__(self, train_matrix, businessRegionEmbedList, place_coords, device=None, seed=0):
        dev = torch.device(device or _device())
        csr = train_matrix.tocsr()  # as stored (never reordered in place: `tocsr()` of a CSR matrix is the caller's object)
        self.num_poi = csr.shape[1]
        self.indptr = np.asarray(csr.indptr, dtype=np.int64)
        self.indices = torch.from_numpy(np.asarray(csr.indices, dtype=np.int64)).to(dev)
        self.region = torch.from_numpy(np.asarray(businessRegionEmbedList, dtype=np.int64)).to(dev)
        self.coords = torch.from_numpy(np.asarray(place_coords, dtype=np.float64)).to(dev)
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(seed)
        self.dev = dev
        self._visited = torch.zeros(self.num_poi, dtype=torch.bool, device=dev)
        # centred float32 coordinates (float64 midpoint subtracted first, like model.set_catalog): what the kernels difference
        c = np.asarray(place_coords, dtype=np.float64)
        self.center = ((c[:, 0].min() + c[:, 0].max()) / 2, (c[:, 1].min() + c[:, 1].max()) / 2)
        self.coords32 = torch.from_numpy((c - np.array(self.center)).astype(np.float32)).to(dev)
        self.region32 = self.region.to(torch.int32)
        self._indptr_dev = torch.from_numpy(self.indptr).to(dev)
        # region id and centred coordinates of every CSR entry: a user's history side data is then a slice (nais_train_users)
        self.entry_region = self.region[self.indices].contiguous()
        self.entry_coords = self.coords32[self.indices].contiguous()

    def multi_user_batch(self, uids, negative_num: int, seed: int = 0):
        """One training batch over MANY users (SURVEY.md §8 f1) as an `ops.SegmentedPairs`: for every user all positives, each
        followed by `negative_num` negatives drawn on the device uniformly without replacement from the POIs outside the
        user's history (the distribution of batches.py:76-80), labels [1, 0..0] interleaved like the reference — but every
        user's history is stored ONCE (the kernels index it per row) and no distance tensor exists (the kernels difference
        the centred coordinates).  `seed` keys the counter-based sampler: same seed, same batch."""
        from . import ops
        uids = np.asarray(uids, dtype=np.int64)
        H = self.indptr[uids + 1] - self.indptr[uids]
        # where every history entry of the batch sits in the CSR (host arithmetic: the indptr is here), riding in the same upload
        seg_off = np.concatenate([[0], np.cumsum(H)])
        src_h = np.repeat(self.indptr[uids] - seg_off[:-1], H) + np.arange(int(seg_off[-1]), dtype=np.int64)
        st = ops.segment_structure(H, (negative_num + 1) * H, self.dev, extra=[(src_h, np.int64)])
        hist = self.indices[st["extra"][0]]
        tgt, label, treg, tcoords = ops.sample_batch(hist, st, negative_num, self.num_poi, seed, self.region32, self.coords32)
        fields = {k: st[k] for k in ("seg_offsets", "row_offsets", "seg_cell_offsets", "tile_seg", "tile_row0", "n_seg", "B", "n_tiles",
                                     "n_cells", "max_hist", "host_row_offsets")}
        return ops.SegmentedPairs(hist=hist, hreg=self.region[hist], hist_coords=self.coords32[hist].contiguous(), tgt=tgt, treg=treg,
                                  tgt_coords=tcoords, label=label, center=self.center, **fields)

    def batch(self, uid: int, negative_num: int):
        """-> (user_history [B,H], train_data [B], train_label [B], user_history_region [B,H], train_data_region [B],
        target_lat_long [B,H,2])  with B = H * (negative_num + 1)."""
        a, b = int(self.indptr[uid]), int(self.indptr[uid + 1])
        pos = self.indices[a:b]
        H = b - a
        pos = pos[torch.randperm(H, device=self.dev, generator=self.gen)]
        m = H * negative_num
        # uniform without replacement over the non-visited POIs: a random permutation with the visited ones removed
        perm = torch.randperm(self.num_poi, device=self.dev, generator=self.gen)[: m + H]
        self._visited[pos] = True
        neg = perm[~self._visited[perm]][:m]
        self._visited[pos] = False
        tgt = torch.cat((pos.view(-1, 1), neg.view(-1, negative_num)), dim=1).reshape(-1)
        label = torch.zeros(H, negative_num + 1, device=self.dev)
        label[:, 0] = 1.0
        hist = pos.unsqueeze(0).expand(tgt.numel(), H).contiguous()
        ll = (self.coords[tgt].unsqueeze(1) - self.coords[pos].unsqueeze(0)).abs().to(torch.float32).contiguous()
        return hist, tgt, label.reshape(-1), self.region[hist], self.region[tgt], ll
