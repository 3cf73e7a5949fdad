"""Multi-GPU plumbing (one process per GPU, `torch.distributed`): range-sharded full-rank evaluation and data-parallel
training.

Evaluation.  The (user, candidate) pairs are independent — the beta-softmax normalises over the user's *history*, not over
candidates (SURVEY.md §8e) — so the catalogue is split into contiguous POI ranges (and, when the catalogue is too small
for `world` useful shards, the user batch into slices: `grid_shape`); each rank scores its users against its own range
with the fused kernel (against a `nais_fullrank_prepare` plan of its range, built once per model), keeps a local top-k as
packed 8-byte ranking keys, and ONE collective per user batch exchanges them: `all_gather_into_tensor` of [U, k] int64 =
U*k*8*world bytes per rank.  The gathered [world, U, k] buffer is merged in place by `nais_topk_merge_keys` (same order rule
as the single-GPU top-k, so results are identical to one GPU).

Training.  Data parallel over rows: dense all-reduce of the gradients (`allreduce_gradients`), or — for catalogues where the
dense tables are hundreds of MB — the touched-row exchange of `SparseRowExchange` (all-gather of (row id, gradient row) lists
and a row-sparse Adagrad on the union, SURVEY.md §8e 'Train partitioning').

The reference has no distributed code at all (SURVEY.md §5); this module is new.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import ops


def shard_range(n: int, rank: int, world: int, align: int = 128) -> Tuple[int, int]:
    """Contiguous POI range of `rank`: boundaries at multiples of `align` (the scorer's candidate tile) so no tile
    straddles two ranks; the last rank takes the remainder."""
    per = (n + world - 1) // world
    per = (per + align - 1) // align * align
    lo = min(n, rank * per)
    hi = min(n, lo + per) if rank < world - 1 else n
    return lo, max(lo, hi)


def gather_keys(keys: torch.Tensor, world: int) -> torch.Tensor:
    """ONE all-gather of the per-rank key lists [U, k] int64 -> [world, U, k] (rank-major)."""
    U, k = keys.shape
    out = torch.empty(world * U, k, dtype=keys.dtype, device=keys.device)
    dist.all_gather_into_tensor(out, keys.contiguous())
    return out.view(world, U, k)


def grid_shape(n_items: int, world: int, min_shard_pois: int) -> Tuple[int, int]:
    """(catalogue shards, user slices) with shards * slices == world: the catalogue is split as far as every shard keeps
    at least `min_shard_pois` POIs, the remaining factor splits the users of a batch.  A rank packs the operand image of
    every user it scores, whatever its catalogue range is, so thin shards pay that cost `world` times (C2's 40k POIs on 8
    GPUs: 12 % of a step); a 1M-POI catalogue is sharded 8 ways as SURVEY.md §8e prescribes."""
    gc = 1
    for d in range(1, world + 1):
        if world % d == 0 and (d == 1 or n_items // d >= min_shard_pois):
            gc = d
    return gc, world // gc


def _merge_cuda(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    return ops.topk_merge_keys(keys)


class ShardedRanker:
    """predict_topk over a range-sharded catalogue (x user-sliced batches when the catalogue is small, `grid_shape`).
    `local_topk` / `merge` / `slice_users` are injectable so the host-side logic can be exercised with the gloo backend on
    CPU (tests/test_distributed_cpu.py); the defaults are the CUDA ops.  rank = user_slice * catalogue_shards + shard.

    local_topk(users, k, lo, hi, precision) -> keys [U, k] int64, or (score [U,k], id [U,k]) which is packed here
    merge(keys [L, U, k]) -> (score [U, k], id [U, k])

    Geo re-ranking (`topk(..., geo=(a, b, alpha))`) adds one step before the local top-k: every rank takes the power-law
    maximum M_u over its own range, and ONE all_reduce(MAX) of a [gu * per] vector — each rank fills only its own user slice,
    -inf elsewhere — leaves every rank the maximum over the whole catalogue for the users it scores.
    local_logmax(users, lo, hi, a, b) -> M [U] float32
    local_topk(users, k, lo, hi, precision, geo: ops.GeoMix) -> as above, ranked by the mix"""

    def __init__(self, model, rank: int = 0, world: int = 1, local_topk: Optional[Callable] = None,
                 merge: Optional[Callable] = None, min_shard_pois: int = 32768, slice_users: Optional[Callable] = None,
                 grid: Optional[Tuple[int, int]] = None, local_logmax: Optional[Callable] = None):
        self.model, self.rank, self.world = model, rank, world
        self.n = model.item_num
        self.gc, self.gu = grid if grid is not None else grid_shape(self.n, world, min_shard_pois)
        if self.gc * self.gu != world:
            raise ValueError(f"grid {self.gc} x {self.gu} does not cover {world} ranks")
        self.rc, self.ru = rank % self.gc, rank // self.gc
        self.lo, self.hi = shard_range(self.n, self.rc, self.gc)
        self._local = local_topk or self._cuda_local
        self._logmax = local_logmax or self._cuda_logmax
        self._merge = merge or _merge_cuda
        self._slice = slice_users or (lambda users, u0, u1: users.slice(u0, u1))
        self.events = []

    def _cuda_local(self, users, k, lo, hi, precision, geo=None):
        m = self.model
        plan = m.ranking_plan(precision, lo, hi)  # built on the first batch, reused while the weights stand
        return ops.fullrank_topk(m.variant, float(m.beta), m._params(), m._catalog, users, k, lo, hi, True, plan.precision, plan,
                                 return_keys=self.world > 1, geo=geo)  # one GPU: the merge kernel writes score / id itself

    def _cuda_logmax(self, users, lo, hi, a, b):
        return ops.powerlaw_logmax(self.model._catalog, users, a, b, lo, hi, True)

    def _global_logmax(self, users, n_users: int, a: float, b: float) -> torch.Tensor:
        """M_u of this rank's users over the whole catalogue: local maxima, then one all_reduce(MAX) among the ranks that
        score the same users (one vector over every slice; a rank leaves the slices of other ranks at -inf)."""
        m = self._logmax(users, self.lo, self.hi, a, b)
        if self.world == 1:
            return m
        u0, u1, per = self.user_range(n_users)
        full = torch.full((self.gu * per,), float("-inf"), dtype=torch.float32, device=m.device)
        full[self.ru * per:self.ru * per + (u1 - u0)] = m
        dist.all_reduce(full, op=dist.ReduceOp.MAX)
        return full[self.ru * per:self.ru * per + (u1 - u0)].contiguous()

    def kernel_name(self, precision: str) -> str:
        return {"fp32": "fullrank_fp32_kernel"}.get(precision, "fullrank_tc_kernel")

    @property
    def parallelism(self) -> str:
        return (f"{self.gc} catalogue range shard(s) x {self.gu} user slice(s), one all-gather of the packed top-k keys" +
                (" + on-device merge" if self.gc > 1 else ""))

    @property
    def last_kernel_ms(self) -> Optional[float]:
        if not self.events:
            return None
        a, b = self.events[-1]
        b.synchronize()
        return a.elapsed_time(b)

    def user_range(self, n_users: int) -> Tuple[int, int, int]:
        """(u0, u1, per): this rank scores users [u0, u1) of a batch; every slice is padded to `per` rows for the gather."""
        per = (n_users + self.gu - 1) // self.gu
        u0 = min(n_users, self.ru * per)
        return u0, min(n_users, u0 + per), per

    def _score_and_exchange(self, users, n_users: int, k: int, precision: str, timed: bool, geo=None):
        """`users` = this rank's slice.  Local fused scoring + top-k, then ONE all-gather of the key lists and the
        on-device merge / unpack; every rank returns the lists of the whole batch [n_users, k]."""
        u0, u1, per = self.user_range(n_users)
        if timed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        if geo is None:
            keys = self._local(users, k, self.lo, self.hi, precision)
        else:
            ga, gb, galpha = (float(x) for x in geo)
            logmax = self._global_logmax(users, n_users, ga, gb)
            keys = self._local(users, k, self.lo, self.hi, precision, ops.GeoMix(ga, gb, galpha, logmax))
        if timed:
            b.record()
            self.events = [(a, b)]
        if self.world == 1:
            return keys if isinstance(keys, tuple) else self._merge(keys.unsqueeze(0))
        if isinstance(keys, tuple):
            keys = ops.lists_to_keys(*keys)
        if keys.shape[0] < per:  # last slice: pad with "no entry" rows (key 0)
            keys = torch.cat([keys, keys.new_zeros((per - keys.shape[0], k))])
        g = gather_keys(keys, self.world)                      # [world, per, k], rank = slice * gc + shard
        if self.gu == 1:
            return self._merge(g)
        if self.gc == 1:  # user slices only: the gathered buffer IS the batch in user order; one unpack of [gu * per, k]
            s_, i_ = self._merge(g.view(1, self.gu * per, k))
            return s_[:n_users], i_[:n_users]
        outs = [self._merge(g[s * self.gc:(s + 1) * self.gc]) for s in range(self.gu)]  # one [gc, per, k] block per slice
        return torch.cat([o[0] for o in outs])[:n_users], torch.cat([o[1] for o in outs])[:n_users]

    def topk(self, users, k: int, precision: str = "auto", geo: Optional[Tuple[float, float, float]] = None):
        """`users`: the whole batch (DeviceUsers), resident on every rank.  `geo` = (a, b, alpha): rank by the power-law
        mix of `powerlaw.fused_rerank_topk` (the scores returned are the mixed values)."""
        timed = torch.cuda.is_available() and users.offsets.is_cuda
        n_users = getattr(users, "n_users", None)
        if self.gu > 1:
            u0, u1, _ = self.user_range(n_users)
            users = self._slice(users, u0, u1)
        return self._score_and_exchange(users, n_users, k, precision, timed, geo)

    def topk_host(self, indptr: torch.Tensor, items: torch.Tensor, k: int, precision: str = "auto"):
        """End-to-end call: pinned host CSR -> device (only this rank's user slice), rank, top-k lists of the whole batch
        back on the host (sigmoid scores like `forward`, int64 ids)."""
        m = self.model
        dev = next(m.parameters()).device
        n_users = indptr.numel() - 1
        u0, u1, _ = self.user_range(n_users)
        a, b = int(indptr[u0]), int(indptr[u1])
        ip = indptr[u0:u1 + 1].to(dev, non_blocking=True) - a
        it = items[a:b].to(dev, non_blocking=True)
        cat = m._catalog
        users = ops.DeviceUsers(ip, it.to(torch.int32), cat.region[it] if cat.region is not None else None,
                                cat.coords[it].contiguous() if cat.coords is not None else None, u1 - u0, b - a)
        s, i = self._score_and_exchange(users, n_users, k, precision, True)
        s_h = torch.sigmoid(s).to("cpu", non_blocking=True)
        i_h = i.to(torch.int64).to("cpu", non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return s_h, i_h


def allreduce_gradients(model, world: int) -> None:
    """Data-parallel training: average dense gradients across ranks (MLP grads ~17 KB + embedding tables; SURVEY.md
    §8e 'Train partitioning').  One flat bucket -> one NCCL all-reduce."""
    if world <= 1:
        return
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    if flat.is_cuda:
        dist.all_reduce(flat, op=dist.ReduceOp.AVG)  # NCCL averages in the collective
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)  # gloo (CPU tests) has no AVG
        flat.div_(world)
    torch._foreach_copy_(grads, [v.view_as(g) for v, g in zip(flat.split([g.numel() for g in grads]), grads)])


class SparseRowExchange:
    """Data-parallel training step for catalogues where the dense embedding gradients are hundreds of MB (C4: 2 x 128 MB at 1M
    POIs) — SURVEY.md §8e 'Train partitioning': every rank runs forward + backward on ITS rows with row-compacted table gradients
    (only the touched rows exist), the ranks all-gather their (row id, gradient row) lists, and every rank applies the same
    row-sparse Adagrad step to the union (`nais_rows_adagrad`: equal ids summed in rank-major list order, so the replicas stay
    bit-identical).  The attention-MLP / dist-layer gradients (17 KB) are all-reduced densely and stepped by `optimizer.step()`.

    Loss = mean BCE over the GLOBAL batch (every rank's rows weighted 1 / (world * local rows)), or `row_weight / world`.
    With weight_decay = lr_decay = 0 (run.py:833) the result equals one dense torch.optim.Adagrad step on the concatenated batch."""

    def __init__(self, model, optimizer: torch.optim.Adagrad, world: int = 1):
        self.model, self.opt, self.world = model, optimizer, world
        P = model._params()
        dev = next(model.parameters()).device
        self.remaps = {n: torch.zeros(P[n].shape[0], dtype=torch.int32, device=dev) for n in ops._TABLES if n in P}
        self.last_bytes = 0  # bytes this rank received in the last exchange

    def _hyper(self, P):
        group_of = {id(p): g for g in self.opt.param_groups for p in g["params"]}
        sums, lr, eps = {}, None, None
        for name in self.remaps:
            g = group_of[id(P[name])]
            if g["weight_decay"] != 0 or g["lr_decay"] != 0 or g.get("maximize", False):
                raise RuntimeError("row-sparse Adagrad equals the dense step only for weight_decay = lr_decay = 0")
            lr, eps = g["lr"], g["eps"]
            st = self.opt.state[P[name]]
            if "sum" not in st:  # (torch creates the state in the optimizer's constructor; be safe for exotic subclasses)
                st["sum"] = torch.full_like(P[name], g.get("initial_accumulator_value", 0.0))
                st["step"] = torch.tensor(0.0)
            sums[name] = st["sum"]
        return sums, lr, eps

    def exchange(self, ids: torch.Tensor, rows: torch.Tensor):
        """all-gather of one table's (ids, rows): -> (ids [n] in rank-major list order, rows [n, w]) of every rank."""
        if self.world == 1:
            return ids, rows
        n = torch.tensor([ids.numel()], device=ids.device, dtype=torch.int64)
        counts = torch.empty(self.world, device=ids.device, dtype=torch.int64)
        dist.all_gather_into_tensor(counts, n)
        counts = counts.cpu()
        cap, w = int(counts.max()), rows.shape[1]
        pi = ids.new_full((cap,), -1)
        pi[:ids.numel()] = ids
        pr = rows.new_zeros((cap, w))
        pr[:ids.numel()] = rows
        gi = torch.empty(self.world * cap, device=ids.device, dtype=ids.dtype)
        gr = torch.empty(self.world * cap, w, device=ids.device, dtype=rows.dtype)
        dist.all_gather_into_tensor(gi, pi)
        dist.all_gather_into_tensor(gr, pr)
        self.last_bytes += gi.numel() * 8 + gr.numel() * 4
        valid = gi >= 0
        return gi[valid], gr[valid]

    def step(self, label, hist, tgt=None, hreg=None, treg=None, aux=None, row_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
        m = self.model
        P = m._params()
        sums, lr, eps = self._hyper(P)
        pp = getattr(m, "pairs_precision", "auto")
        drop = (0.0, 0, pp)
        self.opt.zero_grad(set_to_none=True)
        with torch.no_grad():
            score, row_sum, parts, mask = ops.pairs_forward_raw(m.variant, float(m.beta), P, hist, tgt, hreg, treg, aux, drop)
        s = score.detach().requires_grad_(True)
        if row_weight is None:
            loss = m.loss_func(torch.sigmoid(s), label) / self.world
        else:
            loss = (torch.nn.functional.binary_cross_entropy(torch.sigmoid(s), label, reduction="none") * row_weight).sum() / self.world
        loss.backward()
        self.last_bytes = 0
        with torch.no_grad():
            G, sparse = ops.pairs_backward_compact(m.variant, float(m.beta), P, hist, tgt, hreg, treg, aux, row_sum, parts, s.grad,
                                                   self.remaps, drop, act_mask=mask)
            for name, (ids, rows) in sparse.items():
                gi, gr = self.exchange(ids, rows)
                order = torch.sort(gi, stable=True).indices  # key order; equal ids keep their rank-major order
                ops.rows_adagrad(gi[order], gr[order], P[name], sums[name], lr, eps)
            if self.world > 1:
                flat = torch.cat([g.reshape(-1) for g in G.values()])
                dist.all_reduce(flat, op=dist.ReduceOp.SUM)
                o = 0
                for g in G.values():
                    g.copy_(flat[o:o + g.numel()].view_as(g))
                    o += g.numel()
        for name, grad in G.items():
            P[name].grad = grad.to(P[name].dtype)
        self.opt.step()  # MLP / dist layer; the tables have no .grad
        m._plan_epoch = getattr(m, "_plan_epoch", 0) + 1
        total = loss.detach().clone()
        if self.world > 1:
            dist.all_reduce(total, op=dist.ReduceOp.SUM)
        return total
