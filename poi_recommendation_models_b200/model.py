"""Drop-in mirror of the reference's NAIS classes (`/root/reference/model.py`), backed by libnais_b200.so.

Same class names, constructor arguments, `forward` / `attention_network` / `get_mask` / `loss_function` signatures,
attributes (`embed_size, item_num, beta, hidden_size, loss_func`) and `state_dict` keys as

    NAIS_basic                                   model.py:8-97
    NAIS_regionEmbedding                         model.py:99-187
    NAIS_region_distance_Embedding               model.py:189-304     <- the parity target (run.py:222)
    NAIS_distance_Embedding                      model.py:306-408
    NAIS_region_distance_disentangled_Embedding  model.py:410-541

so `torch.optim.Adagrad(model.parameters())`, `model.train()/eval()`, `torch.save(model)`, and loading a reference
checkpoint's `state_dict` all work unchanged.  The submodules are created and initialised in the reference's order, so
the same `torch.manual_seed` gives the same initial weights.  What differs is what runs: `attention_network` is one
fused CUDA kernel (plus hand-written backward kernels) instead of ~25 ATen ops, and there is an additional
`predict_topk` entry that replaces the whole per-user loop of `validation.py:84-127`.

There is no CPU path: calling a model whose parameters or inputs are not on a CUDA device raises.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import ops


class _NAISBase(nn.Module):
    variant = ""
    _dropout_on_l1 = False  # NAIS_basic / NAIS_regionEmbedding apply nn.Dropout() to the L1 output (model.py:71,162)

    # -- shared construction helpers -------------------------------------------------------------------------------
    def _common(self, item_num, embed_size, hidden_size, beta):
        self.DEVICE = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self.embed_size = embed_size
        self.item_num = item_num
        self.beta = beta
        self.hidden_size = hidden_size
        self._catalog: Optional[ops.DeviceCatalog] = None
        self._plans: Dict[tuple, ops.FullrankPlan] = {}
        self._plan_epoch = 0  # bumped by every in-place parameter update torch's version counters do not see
        # which kernels forward / backward run: "auto" = tcgen05 where the shape has them (one branch, D in {16..64}, hid <= 128;
        # backward: hid = 64, D in {32, 64}), else the FP32 CUDA-core kernels; "fp32" / "tc" force one (NaisParams::pairs_precision)
        self.pairs_precision = "auto"

    def _acts(self):
        self.relu = nn.ReLU()
        self.sigmoid = nn.Sigmoid()
        self.loss_func = nn.BCELoss()

    def _init_weight_(self):
        # embeddings N(0, 0.01); Linear biases zero; Linear weights keep torch's default (model.py:219-229)
        for name in ("embed_history", "embed_target", "embed_region", "embed_distance"):
            if hasattr(self, name):
                nn.init.normal_(getattr(self, name).weight, std=0.01)
        for m in self.modules():
            if isinstance(m, nn.Linear) and m.bias is not None:
                m.bias.data.zero_()

    # -- the scorer -------------------------------------------------------------------------------------------------
    def _params(self) -> Dict[str, torch.Tensor]:
        named = dict(self.named_parameters())
        return {n: named[n] for n in ops.VARIANT_PARAMS[self.variant]}

    def _draw_dropout(self) -> Tuple[float, int]:
        """(p, seed) of this call's dropout: relu(drop(attn_layer1(x))) in train mode (model.py:71,162) is fused, with a
        counter-based mask; the seed comes from torch's CPU generator so torch.manual_seed makes a run reproducible (not the
        reference's mask stream).  (0.0, 0) when no dropout applies."""
        if self._dropout_on_l1 and self.training and self.drop.p > 0:
            self.last_dropout_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            return float(self.drop.p), self.last_dropout_seed
        return 0.0, 0

    def _score(self, hist, tgt, hreg=None, treg=None, aux=None) -> torch.Tensor:
        drop_p, seed = self._draw_dropout()
        P = self._params()
        return ops.pairs_score(self.variant, float(self.beta), tuple(P.values()), hist, tgt, hreg, treg, aux, drop_p, seed,
                               getattr(self, "pairs_precision", "auto"))

    def segmented_scores(self, batch: "ops.SegmentedPairs") -> torch.Tensor:
        """`attention_network` over a multi-user batch in the segmented layout (ops.SegmentedPairs: the rows of a user share
        one stored history, distances are formed in the kernel): pre-sigmoid scores [B], differentiable like the per-user
        call.  One step over U users gives exactly the sum of the U single-user gradients (tests/test_gpu_segmented.py).  In train
        mode the dropout classes apply dropout as `attention_network` does (the mask is indexed by the segmented cell)."""
        drop_p, seed = self._draw_dropout()
        P = self._params()
        return ops.pairs_score(self.variant, float(self.beta), tuple(P.values()), batch, None, None, None, None, drop_p, seed,
                               getattr(self, "pairs_precision", "auto"))

    def fused_adagrad_step(self, optimizer: torch.optim.Adagrad, label, hist, tgt=None, hreg=None, treg=None, aux=None,
                           row_weight: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One training step of run.py:248-254 (`zero_grad -> forward -> BCELoss -> backward -> Adagrad.step`) with the
        embedding tables stepped by the row-sparse Adagrad fused into the backward's segment reduce: no dense
        [N, D/2] gradient is zero-filled, written or read, and only the touched rows of the tables and of the optimizer's
        `state['sum']` move.  With the reference's `weight_decay = 0` (run.py:833) this IS the dense step (SURVEY.md §7
        'Dense Adagrad semantic'); other settings raise.  The MLP / dist-layer parameters go through `optimizer.step()` as
        usual.  Returns the loss (same value `loss_func(forward(...), label)` gives).  `hist` may be an ops.SegmentedPairs
        (many users in one step; tgt / hreg / treg / aux then stay None).  Every class takes the one-call path, the two-branch
        disentangled one included (its embed_distance moves in row 0, the only row its forward reads).  `row_weight` [B]: the loss becomes
        sum_b row_weight[b] * BCE_b instead of the batch mean — e.g. 1 / rows(user of b) makes a multi-user step the sum of the
        reference's per-user mean losses (run.py:251)."""
        if not isinstance(optimizer, torch.optim.Adagrad):
            raise RuntimeError("fused_adagrad_step needs torch.optim.Adagrad (run.py:225)")
        P = self._params()
        group_of = {id(p): g for g in optimizer.param_groups for p in g["params"]}
        sums, lr, eps = {}, None, None
        for name in ops._TABLES:
            if name not in P:
                continue
            g = group_of.get(id(P[name]))
            if g is None:
                raise RuntimeError(f"{name} is not in the optimizer")
            if g["weight_decay"] != 0 or g["lr_decay"] != 0 or g.get("maximize", False):
                raise RuntimeError("row-sparse Adagrad equals the dense step only for weight_decay = lr_decay = 0")
            if lr is not None and (lr, eps) != (g["lr"], g["eps"]):
                raise RuntimeError("embedding tables must share lr / eps")
            lr, eps = g["lr"], g["eps"]
            sums[name] = optimizer.state[P[name]]["sum"]
        pp = getattr(self, "pairs_precision", "auto")
        drop = (*self._draw_dropout(), pp)
        # ---- everything in one library call (nais_pairs_train_step) when the step is the reference's: mean / row-weighted BCE,
        # plain Adagrad on every parameter.  `one_call=False` on the model keeps the op-by-op path below (the parity tests compare).
        dense = {n: t for n, t in P.items() if n not in ops._TABLES}
        dgroups = [group_of.get(id(t)) for t in dense.values()]
        if (getattr(self, "one_call", True) and isinstance(pp, str) and type(self.loss_func) is nn.BCELoss
                and self.loss_func.reduction == "mean" and self.loss_func.weight is None and all(g is not None for g in dgroups)
                and all(g["weight_decay"] == 0 and g["lr_decay"] == 0 and not g.get("maximize", False) for g in dgroups)
                and len({(g["lr"], g["eps"]) for g in dgroups}) == 1 and all(t.dtype == torch.float32 for t in P.values())):
            optimizer.zero_grad(set_to_none=True)
            dsum = {n: optimizer.state[t]["sum"] for n, t in dense.items()}
            loss, _ = ops.pairs_train_step(self.variant, float(self.beta), P, sums, dsum, lr, eps, dgroups[0]["lr"], dgroups[0]["eps"],
                                           label, hist, tgt, hreg, treg, aux, row_weight, drop)
            for t in P.values():
                optimizer.state[t]["step"] += 1
            self._plan_epoch = getattr(self, "_plan_epoch", 0) + 1
            return loss[0]
        optimizer.zero_grad(set_to_none=True)
        with torch.no_grad():
            score, row_sum, parts, mask = ops.pairs_forward_raw(self.variant, float(self.beta), P, hist, tgt, hreg, treg, aux, drop)
        s = score.detach().requires_grad_(True)  # dL/dscore through torch's own sigmoid + BCELoss ([B]-sized, exact semantics)
        if row_weight is None:
            loss = self.loss_func(torch.sigmoid(s), label)
        else:
            loss = (nn.functional.binary_cross_entropy(torch.sigmoid(s), label, reduction="none") * row_weight).sum()
        loss.backward()
        with torch.no_grad():
            G = ops.pairs_backward_adagrad(self.variant, float(self.beta), P, sums, lr, eps, hist, tgt, hreg, treg, aux, row_sum,
                                           parts, s.grad, drop, act_mask=mask)
        for name, grad in G.items():
            P[name].grad = grad.to(P[name].dtype)
        optimizer.step()  # the tables have no .grad: torch skips them
        self._plan_epoch = getattr(self, "_plan_epoch", 0) + 1  # the kernel stepped the tables behind torch's version counters
        return loss.detach()

    def train_users(self, optimizer: torch.optim.Adagrad, batcher, uids, negative_num: int, seed: int = 0) -> torch.Tensor:
        """The inner loop of `train_NAIS_region_distance` (run.py:227-255) — for every user: sample `negative_num` negatives per
        positive, forward, BCELoss, backward, Adagrad step — for a whole list of users in ONE library call (`nais_train_users`):
        the same optimizer steps in the same order as `for u in uids: fused_adagrad_step(optimizer, *batcher.multi_user_batch([u],
        negative_num, seed + u))`, bit for bit, without the per-user Python work.  `batcher`: a batches.DeviceBatcher over the
        train matrix.  Every class, the disentangled one included.  In train mode the dropout classes draw one mask seed per
        user with a history, in list order, as `torch.randint(0, 2**62, (n_steps,))`: torch's CPU generator gives the values of
        n_steps single draws, so under the same `torch.manual_seed` the steps are the loop's.  Returns the per-user losses
        [len(uids)] on the device."""
        if not isinstance(optimizer, torch.optim.Adagrad):
            raise RuntimeError("train_users needs torch.optim.Adagrad (run.py:225)")
        if type(self.loss_func) is not nn.BCELoss or self.loss_func.reduction != "mean":
            raise RuntimeError("train_users: the reference's mean BCELoss")
        P = self._params()
        group_of = {id(p): g for g in optimizer.param_groups for p in g["params"]}
        groups = [group_of.get(id(t)) for t in P.values()]
        if any(g is None for g in groups) or any(g["weight_decay"] != 0 or g["lr_decay"] != 0 or g.get("maximize", False) for g in groups):
            raise RuntimeError("train_users: plain Adagrad (weight_decay = lr_decay = 0) on every parameter")
        tg = {(group_of[id(t)]["lr"], group_of[id(t)]["eps"]) for n, t in P.items() if n in ops._TABLES}
        dg = {(group_of[id(t)]["lr"], group_of[id(t)]["eps"]) for n, t in P.items() if n not in ops._TABLES}
        if len(tg) != 1 or len(dg) != 1:
            raise RuntimeError("train_users: the tables / the MLP tensors must each share lr and eps")
        (lr_t, eps_t), (lr_d, eps_d) = next(iter(tg)), next(iter(dg))
        sums = {n: optimizer.state[t]["sum"] for n, t in P.items()}
        hu = np.asarray(uids, dtype=np.int64).reshape(-1)
        has_hist = np.asarray(batcher.indptr)[hu + 1] > np.asarray(batcher.indptr)[hu]
        n_steps = int(has_hist.sum())
        drop_p, drop_seeds = 0.0, None
        if self._dropout_on_l1 and self.training and self.drop.p > 0 and n_steps:
            drawn = torch.randint(0, 2 ** 62, (n_steps,))
            drop_p, drop_seeds = float(self.drop.p), np.zeros(hu.size, dtype=np.uint64)
            drop_seeds[has_hist] = drawn.numpy().astype(np.uint64)
            self.last_dropout_seed = int(drawn[-1])
        optimizer.zero_grad(set_to_none=True)
        has_reg, has_co = "embed_region.weight" in P, ops.VARIANT_DIST[self.variant][0] != ops.DIST_NONE
        losses = ops.train_users(self.variant, float(self.beta), P, sums, sums, lr_t, eps_t, lr_d, eps_d, batcher.indptr, batcher.indices,
                                 batcher.entry_region if has_reg else None, batcher.entry_coords if has_co else None,
                                 batcher.region32 if has_reg else None, batcher.coords32 if has_co else None, uids, negative_num, seed,
                                 getattr(self, "pairs_precision", "auto") if isinstance(getattr(self, "pairs_precision", "auto"), str) else "auto",
                                 center=batcher.center, dropout_p=drop_p, dropout_seeds=drop_seeds)
        for t in P.values():
            optimizer.state[t]["step"] += n_steps
        self._plan_epoch = getattr(self, "_plan_epoch", 0) + 1
        return losses

    def get_mask(self, user_history, target_item):
        return user_history != target_item.reshape([len(target_item), 1])

    def loss_function(self, prediction, label):
        return self.loss_func(prediction, label)

    # -- full-rank ranking (new, additive) -----------------------------------------------------------------------------
    def set_catalog(self, region: Optional[Sequence[int]] = None, coords: Optional[np.ndarray] = None,
                    row_base: int = 0) -> None:
        """Register the per-POI side data once (replaces the `businessRegionEmbedList` and `latlon_mat` arguments of
        validation.py:62): dense region ids [N] and (lat, lon) [N,2].  Coordinates are centred on the bounding-box
        midpoint in float64 before the float32 cast, so in-kernel |dlat|,|dlon| match the reference's float64
        differences to ~1e-8 degrees (run.py:47-54, SURVEY.md §7 'Coordinates')."""
        dev = next(self.parameters()).device
        reg = None if region is None else torch.as_tensor(np.asarray(region), dtype=torch.int32, device=dev)
        crd, center = None, (0.0, 0.0)
        if coords is not None:
            c = np.asarray(coords, dtype=np.float64)
            center = (float((c[:, 0].min() + c[:, 0].max()) / 2), float((c[:, 1].min() + c[:, 1].max()) / 2))
            crd = torch.as_tensor((c - np.array(center)).astype(np.float32), device=dev)
        n = len(reg) if reg is not None else (len(crd) if crd is not None else self.item_num - row_base)
        self._catalog = ops.DeviceCatalog(reg, crd, row_base, n, center)
        self._plans = {}

    def _apply(self, fn, *args, **kwargs):
        # .cuda() / .to(device): the catalogue arrays follow the parameters (a catalogue left behind on another device would
        # reach the kernels as a foreign pointer), and every ranking plan is dropped
        super()._apply(fn, *args, **kwargs)
        cat = getattr(self, "_catalog", None)
        if cat is not None:
            dev = next(self.parameters()).device
            mv = lambda t: None if t is None else t.to(dev)
            self._catalog = ops.DeviceCatalog(mv(cat.region), mv(cat.coords), cat.row_base, cat.n_rows, cat.center)
        self._plans = {}
        return self

    def __getstate__(self):
        st = super().__getstate__() if hasattr(nn.Module, "__getstate__") else self.__dict__.copy()
        st = dict(st)
        st["_plans"] = {}  # derived device buffers (up to hundreds of MB): rebuilt on first use, never pickled
        return st

    def ranking_plan(self, precision: str = "auto", poi_begin: int = 0, poi_end: Optional[int] = None) -> ops.FullrankPlan:
        """The `nais_fullrank_prepare` plan of the current weights for a catalogue range, built on first use and reused until a
        parameter changes (torch's per-tensor version counters + `_plan_epoch`), the catalogue is replaced or the model
        moves: an evaluation (validation.py:69, one frozen model, every user) pays the per-model constants once."""
        if self._catalog is None:
            raise RuntimeError("call set_catalog(region, coords) first")
        P = self._params()
        poi_end = self.item_num if poi_end is None else poi_end
        key = (precision, poi_begin, poi_end, getattr(self, "_plan_epoch", 0), float(self.beta)) + tuple(
            (t.data_ptr(), t._version) for t in P.values())
        plan = self._plans.get((precision, poi_begin, poi_end))
        if plan is None or plan.key != key:
            plan = ops.fullrank_prepare(self.variant, float(self.beta), P, self._catalog, poi_begin, poi_end, precision)
            plan.key = key
            self._plans[(precision, poi_begin, poi_end)] = plan
        return plan

    def make_users(self, indptr, indices) -> ops.DeviceUsers:
        """CSR histories (train_matrix.indptr / .indices, validation.py:86) -> device arrays with region ids and
        centred coordinates of every history item gathered."""
        if self._catalog is None:
            raise RuntimeError("call set_catalog(region, coords) first")
        cat = self._catalog
        dev = next(self.parameters()).device
        off = torch.as_tensor(np.asarray(indptr), dtype=torch.int64, device=dev)
        it = torch.as_tensor(np.asarray(indices), dtype=torch.int64, device=dev)
        if cat.row_base != 0 and (cat.region is not None or cat.coords is not None):
            raise RuntimeError("history gathering needs the full catalogue on this device (row_base == 0)")
        if it.numel() and (int(it.min()) < 0 or int(it.max()) >= self.item_num):  # what nn.Embedding would raise on (host-side: this
            raise IndexError("history item id outside [0, item_num)")              # call builds device arrays from host CSR anyway)
        reg = cat.region[it] if cat.region is not None else None
        crd = cat.coords[it].contiguous() if cat.coords is not None else None
        return ops.DeviceUsers(off, it.to(torch.int32), reg, crd, len(indptr) - 1, int(len(indices)),
                               np.asarray(indptr, dtype=np.int64))

    @torch.no_grad()
    def predict_topk(self, users, k: int, exclude_history: bool = True, poi_begin: int = 0,
                     poi_end: Optional[int] = None, precision: str = "auto") -> Tuple[torch.Tensor, torch.Tensor]:
        """Top-k POIs of [poi_begin, poi_end) for every user: (sigmoid score [U,k] as `forward` would return,
        ids [U,k] int64, -1 padded).  `users` is a DeviceUsers or an (indptr, indices) pair.  One call replaces the
        user loop of validation.py:84-127 (candidates = all - history, chunked forward, cat, topk).  precision: "auto"
        (tensor-core path with its device-side accuracy gate where the shape has one, else FP32), "fp32", "tc_auto",
        "tc_split", "tc_mix", "tc_fast" (ops.resolve_precision, include/nais_b200.h NAIS_PREC_*)."""
        if not isinstance(users, ops.DeviceUsers):
            users = self.make_users(*users)
        plan = self.ranking_plan(precision, poi_begin, poi_end)
        s, i = ops.fullrank_topk(self.variant, float(self.beta), self._params(), self._catalog, users, k, poi_begin,
                                 poi_end, exclude_history, plan.precision, plan)
        return torch.sigmoid(s), i.to(torch.int64)


class NAIS_basic(_NAISBase):
    variant = "basic"
    _dropout_on_l1 = True

    def __init__(self, item_num, embed_size, hidden_size, beta):
        super().__init__()
        self._common(item_num, embed_size, hidden_size, beta)
        self.embed_history = nn.Embedding(item_num, embed_size)
        self.embed_target = nn.Embedding(item_num, embed_size)
        self._acts()
        self.drop = nn.Dropout()
        self.attn_layer1 = nn.Linear(embed_size, hidden_size)
        self.attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self._init_weight_()

    def forward(self, history, target):
        return self.sigmoid(self.attention_network(history, target))

    def attention_network(self, user_history, target_item):
        return self._score(user_history, target_item)


class NAIS_regionEmbedding(_NAISBase):
    variant = "region"
    _dropout_on_l1 = True

    def __init__(self, item_num, embed_size, hidden_size, beta, region_embed_size):
        super().__init__()
        self._common(item_num, embed_size, hidden_size, beta)
        self.embed_history = nn.Embedding(item_num, int(embed_size / 2))
        self.embed_target = nn.Embedding(item_num, int(embed_size / 2))
        self.embed_region = nn.Embedding(region_embed_size, int(embed_size / 2))
        self._acts()
        self.attn_layer1 = nn.Linear(embed_size, hidden_size)
        self.attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self.drop = nn.Dropout()
        self._init_weight_()

    def forward(self, history, target, history_region, target_region):
        return self.sigmoid(self.attention_network(history, target, history_region, target_region))

    def attention_network(self, user_history, target_item, history_region, target_region):
        return self._score(user_history, target_item, history_region, target_region)


class NAIS_region_distance_Embedding(_NAISBase):
    variant = "region_distance"

    def __init__(self, item_num, embed_size, hidden_size, beta, region_embed_size, dist_embed_size):
        super().__init__()
        self._common(item_num, embed_size, hidden_size, beta)
        self.embed_history = nn.Embedding(item_num, int(embed_size / 2))
        self.embed_target = nn.Embedding(item_num, int(embed_size / 2))
        self.embed_region = nn.Embedding(region_embed_size, int(embed_size / 2))
        self.embed_distance = nn.Embedding(dist_embed_size, embed_size)  # allocated, never read (model.py:204)
        self._acts()
        self.tanh = nn.Tanh()
        self.attn_layer1 = nn.Linear(embed_size + 2, hidden_size)
        self.attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self.dist_layer = nn.Linear(2, 2)
        self._init_weight_()

    def forward(self, history, target, history_region, target_region, target_lat_long):
        return self.sigmoid(self.attention_network(history, target, history_region, target_region, target_lat_long))

    def attention_network(self, user_history, target_item, history_region, target_region, target_lat_long_tensor):
        return self._score(user_history, target_item, history_region, target_region, target_lat_long_tensor)


class NAIS_distance_Embedding(_NAISBase):
    variant = "distance"

    def __init__(self, item_num, embed_size, hidden_size, beta, region_embed_size, dist_embed_size):
        super().__init__()
        self._common(item_num, embed_size, hidden_size, beta)
        self.embed_history = nn.Embedding(item_num, embed_size)
        self.embed_target = nn.Embedding(item_num, embed_size)
        self._acts()
        self.attn_layer1 = nn.Linear(embed_size + 2, hidden_size)
        self.attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self.dist_layer = nn.Linear(2, 2)
        self._init_weight_()

    def forward(self, history, target, history_region, target_region, target_distance):
        # region arguments are accepted and ignored, as in the reference (model.py:340-353)
        return self.sigmoid(self.attention_network(history, target, target_distance))

    def attention_network(self, user_history, target_item, target_lat_long_tensor):
        return self._score(user_history, target_item, None, None, target_lat_long_tensor)


class NAIS_region_distance_disentangled_Embedding(_NAISBase):
    variant = "disentangled"

    def __init__(self, item_num, embed_size, hidden_size, beta, region_embed_size, dist_embed_size):
        super().__init__()
        self._common(item_num, embed_size, hidden_size, beta)
        self.embed_history = nn.Embedding(item_num, embed_size)
        self.embed_target = nn.Embedding(item_num, embed_size)
        self.embed_region = nn.Embedding(region_embed_size, embed_size)
        self.embed_distance = nn.Embedding(dist_embed_size, embed_size)
        self._acts()
        self.attn_layer1 = nn.Linear(embed_size, hidden_size)
        self.attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self.region_attn_layer1 = nn.Linear(embed_size, hidden_size)
        self.region_attn_layer2 = nn.Linear(hidden_size, 1, bias=False)
        self._init_weight_()

    def forward(self, history, target, history_region, target_region, target_distance):
        return self.sigmoid(self.attention_network(history, target, history_region, target_region, target_distance))

    def attention_network(self, user_history, target_item, history_region, target_region, target_distance):
        return self._score(user_history, target_item, history_region, target_region, target_distance)


CLASSES = {c.variant: c for c in (NAIS_basic, NAIS_regionEmbedding, NAIS_region_distance_Embedding,
                                  NAIS_distance_Embedding, NAIS_region_distance_disentangled_Embedding)}
