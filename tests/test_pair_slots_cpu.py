"""Which tensor of each model variant goes into which slot of NaisParams, NaisGrads, NaisAdagrad and NaisDenseAdagrad.  A slot
that is missed fails silently on the device (a NULL gradient pointer is a gradient never computed, a wrong optimizer-state
pointer corrupts the state), so the fill functions of ops.py are pinned here, on CPU tensors: every struct is described as
field -> parameter name and compared with the tables below."""
import pytest
import torch

from poi_recommendation_models_b200 import ops

N, R, K, HID = 50, 7, 3, 6
# [rows, width] of the tables and the first attention layer of each variant (every other tensor: the defaults of _params)
SHAPES = {
    "basic": {"embed_history.weight": (N, 8), "embed_target.weight": (N, 8), "attn_layer1.weight": (HID, 8)},
    "region": {"embed_history.weight": (N, 4), "embed_target.weight": (N, 4), "embed_region.weight": (R, 4),
               "attn_layer1.weight": (HID, 8)},
    "region_distance": {"embed_history.weight": (N, 4), "embed_target.weight": (N, 4), "embed_region.weight": (R, 4),
                        "attn_layer1.weight": (HID, 10), "dist_layer.weight": (1, 2), "dist_layer.bias": (1,)},
    "distance": {"embed_history.weight": (N, 8), "embed_target.weight": (N, 8), "attn_layer1.weight": (HID, 10),
                 "dist_layer.weight": (1, 2), "dist_layer.bias": (1,)},
    "disentangled": {"embed_history.weight": (N, 8), "embed_target.weight": (N, 8), "embed_region.weight": (R, 8),
                     "embed_distance.weight": (K, 8), "attn_layer1.weight": (HID, 8), "region_attn_layer1.weight": (HID, 8),
                     "region_attn_layer1.bias": (HID,), "region_attn_layer2.weight": (1, HID)},
}

# Non-NULL pointer fields and the scalar fields of each struct.  "rows:<table>" / "remap:<table>" are the row-compacted gradient
# rows and the remap of a table; "ws" is the workspace the presorting forward fills in for every table the backward reduces.
# The fused Adagrad backward fills NaisGrads exactly as the backward without tables ("grads_no_tables").
EXPECTED = {
    "basic": {
        "params": {"beta": 0.5, "branch[0].b1": "attn_layer1.bias", "branch[0].hist_poi": "embed_history.weight",
            "branch[0].tgt_poi": "embed_target.weight", "branch[0].w1": "attn_layer1.weight",
            "branch[0].w2": "attn_layer2.weight", "branch[0].w_poi": 8, "branch[0].w_reg": 0, "branch[1].w_poi": 0,
            "branch[1].w_reg": 0, "dist_buckets": 1, "dist_mode": 0, "dist_scale": 0.0, "hid": 6, "item_num": 50,
            "n_branch": 1, "region_num": 0},
        "adagrad": {"eps": 0.25, "lr": 0.5, "sum_hist_poi[0]": "embed_history.weight",
            "sum_tgt_poi[0]": "embed_target.weight"},
        "dense_adagrad": {"eps": 0.0625, "lr": 0.125, "sum_b1": "attn_layer1.bias",
            "sum_w1": "attn_layer1.weight", "sum_w2": "attn_layer2.weight"},
        "grads_tables": {"b1[0]": "attn_layer1.bias", "hist_poi[0]": "embed_history.weight",
            "tgt_poi[0]": "embed_target.weight", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_no_tables": {"b1[0]": "attn_layer1.bias", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_compact": {"b1[0]": "attn_layer1.bias", "hist_poi[0]": "rows:embed_history.weight",
            "remap_hist_poi[0]": "remap:embed_history.weight", "remap_tgt_poi[0]": "remap:embed_target.weight",
            "tgt_poi[0]": "rows:embed_target.weight", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_presort": {"hist_poi[0]": "ws", "tgt_poi[0]": "ws"},
    },
    "region": {
        "params": {"beta": 0.5, "branch[0].b1": "attn_layer1.bias", "branch[0].hist_poi": "embed_history.weight",
            "branch[0].hist_reg": "embed_region.weight", "branch[0].tgt_poi": "embed_target.weight",
            "branch[0].tgt_reg": "embed_region.weight", "branch[0].w1": "attn_layer1.weight",
            "branch[0].w2": "attn_layer2.weight", "branch[0].w_poi": 4, "branch[0].w_reg": 4, "branch[1].w_poi": 0,
            "branch[1].w_reg": 0, "dist_buckets": 1, "dist_mode": 0, "dist_scale": 0.0, "hid": 6, "item_num": 50,
            "n_branch": 1, "region_num": 7},
        "adagrad": {"eps": 0.25, "lr": 0.5, "sum_hist_poi[0]": "embed_history.weight",
            "sum_reg[0]": "embed_region.weight", "sum_tgt_poi[0]": "embed_target.weight"},
        "dense_adagrad": {"eps": 0.0625, "lr": 0.125, "sum_b1": "attn_layer1.bias",
            "sum_w1": "attn_layer1.weight", "sum_w2": "attn_layer2.weight"},
        "grads_tables": {"b1[0]": "attn_layer1.bias", "hist_poi[0]": "embed_history.weight", "reg[0]": "embed_region.weight",
            "tgt_poi[0]": "embed_target.weight", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_no_tables": {"b1[0]": "attn_layer1.bias", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_compact": {"b1[0]": "attn_layer1.bias", "hist_poi[0]": "rows:embed_history.weight",
            "reg[0]": "rows:embed_region.weight", "remap_hist_poi[0]": "remap:embed_history.weight",
            "remap_reg[0]": "remap:embed_region.weight", "remap_tgt_poi[0]": "remap:embed_target.weight",
            "tgt_poi[0]": "rows:embed_target.weight", "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_presort": {"hist_poi[0]": "ws", "reg[0]": "ws", "tgt_poi[0]": "ws"},
    },
    "region_distance": {
        "params": {"beta": 0.5, "branch[0].b1": "attn_layer1.bias", "branch[0].hist_poi": "embed_history.weight",
            "branch[0].hist_reg": "embed_region.weight", "branch[0].tgt_poi": "embed_target.weight",
            "branch[0].tgt_reg": "embed_region.weight", "branch[0].w1": "attn_layer1.weight",
            "branch[0].w2": "attn_layer2.weight", "branch[0].w_poi": 4, "branch[0].w_reg": 4, "branch[1].w_poi": 0,
            "branch[1].w_reg": 0, "dist_b": "dist_layer.bias", "dist_buckets": 1, "dist_mode": 1, "dist_scale": 100.0,
            "dist_w": "dist_layer.weight", "hid": 6, "item_num": 50, "n_branch": 1, "region_num": 7},
        "adagrad": {"eps": 0.25, "lr": 0.5, "sum_hist_poi[0]": "embed_history.weight",
            "sum_reg[0]": "embed_region.weight", "sum_tgt_poi[0]": "embed_target.weight"},
        "dense_adagrad": {"eps": 0.0625, "lr": 0.125, "sum_b1": "attn_layer1.bias",
            "sum_dist_b": "dist_layer.bias", "sum_dist_w": "dist_layer.weight", "sum_w1": "attn_layer1.weight",
            "sum_w2": "attn_layer2.weight"},
        "grads_tables": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "hist_poi[0]": "embed_history.weight", "reg[0]": "embed_region.weight", "tgt_poi[0]": "embed_target.weight",
            "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_no_tables": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_compact": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "hist_poi[0]": "rows:embed_history.weight", "reg[0]": "rows:embed_region.weight",
            "remap_hist_poi[0]": "remap:embed_history.weight", "remap_reg[0]": "remap:embed_region.weight",
            "remap_tgt_poi[0]": "remap:embed_target.weight", "tgt_poi[0]": "rows:embed_target.weight",
            "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_presort": {"hist_poi[0]": "ws", "reg[0]": "ws", "tgt_poi[0]": "ws"},
    },
    "distance": {
        "params": {"beta": 0.5, "branch[0].b1": "attn_layer1.bias", "branch[0].hist_poi": "embed_history.weight",
            "branch[0].tgt_poi": "embed_target.weight", "branch[0].w1": "attn_layer1.weight",
            "branch[0].w2": "attn_layer2.weight", "branch[0].w_poi": 8, "branch[0].w_reg": 0, "branch[1].w_poi": 0,
            "branch[1].w_reg": 0, "dist_b": "dist_layer.bias", "dist_buckets": 1, "dist_mode": 1, "dist_scale": 1000.0,
            "dist_w": "dist_layer.weight", "hid": 6, "item_num": 50, "n_branch": 1, "region_num": 0},
        "adagrad": {"eps": 0.25, "lr": 0.5, "sum_hist_poi[0]": "embed_history.weight",
            "sum_tgt_poi[0]": "embed_target.weight"},
        "dense_adagrad": {"eps": 0.0625, "lr": 0.125, "sum_b1": "attn_layer1.bias",
            "sum_dist_b": "dist_layer.bias", "sum_dist_w": "dist_layer.weight", "sum_w1": "attn_layer1.weight",
            "sum_w2": "attn_layer2.weight"},
        "grads_tables": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "hist_poi[0]": "embed_history.weight", "tgt_poi[0]": "embed_target.weight", "w1[0]": "attn_layer1.weight",
            "w2[0]": "attn_layer2.weight"},
        "grads_no_tables": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_compact": {"b1[0]": "attn_layer1.bias", "dist_b": "dist_layer.bias", "dist_w": "dist_layer.weight",
            "hist_poi[0]": "rows:embed_history.weight", "remap_hist_poi[0]": "remap:embed_history.weight",
            "remap_tgt_poi[0]": "remap:embed_target.weight", "tgt_poi[0]": "rows:embed_target.weight",
            "w1[0]": "attn_layer1.weight", "w2[0]": "attn_layer2.weight"},
        "grads_presort": {"hist_poi[0]": "ws", "tgt_poi[0]": "ws"},
    },
    "disentangled": {
        "params": {"beta": 0.5, "branch[0].b1": "attn_layer1.bias", "branch[0].hist_poi": "embed_history.weight",
            "branch[0].tgt_poi": "embed_target.weight", "branch[0].w1": "attn_layer1.weight",
            "branch[0].w2": "attn_layer2.weight", "branch[0].w_poi": 8, "branch[0].w_reg": 0,
            "branch[1].b1": "region_attn_layer1.bias", "branch[1].hist_reg": "embed_region.weight",
            "branch[1].tgt_reg": "embed_region.weight", "branch[1].w1": "region_attn_layer1.weight",
            "branch[1].w2": "region_attn_layer2.weight", "branch[1].w_poi": 0, "branch[1].w_reg": 8, "dist_buckets": 1,
            "dist_embed": "embed_distance.weight", "dist_mode": 2, "dist_scale": 0.0, "hid": 6, "item_num": 50, "n_branch": 2,
            "region_num": 7},
        "adagrad": {"eps": 0.25, "lr": 0.5, "sum_hist_poi[0]": "embed_history.weight",
            "sum_reg[1]": "embed_region.weight", "sum_tgt_poi[0]": "embed_target.weight"},
        "dense_adagrad": {"eps": 0.0625, "lr": 0.125, "sum_b1": "attn_layer1.bias",
            "sum_dist_embed": "embed_distance.weight", "sum_region_b1": "region_attn_layer1.bias",
            "sum_region_w1": "region_attn_layer1.weight", "sum_region_w2": "region_attn_layer2.weight",
            "sum_w1": "attn_layer1.weight", "sum_w2": "attn_layer2.weight"},
        "grads_tables": {"b1[0]": "attn_layer1.bias", "b1[1]": "region_attn_layer1.bias",
            "dist_embed": "embed_distance.weight", "hist_poi[0]": "embed_history.weight", "reg[1]": "embed_region.weight",
            "tgt_poi[0]": "embed_target.weight", "w1[0]": "attn_layer1.weight", "w1[1]": "region_attn_layer1.weight",
            "w2[0]": "attn_layer2.weight", "w2[1]": "region_attn_layer2.weight"},
        "grads_no_tables": {"b1[0]": "attn_layer1.bias", "b1[1]": "region_attn_layer1.bias",
            "dist_embed": "embed_distance.weight", "w1[0]": "attn_layer1.weight", "w1[1]": "region_attn_layer1.weight",
            "w2[0]": "attn_layer2.weight", "w2[1]": "region_attn_layer2.weight"},
    },
}


def _params(variant):
    s = dict(SHAPES[variant])
    s.setdefault("attn_layer1.bias", (HID,))
    s.setdefault("attn_layer2.weight", (1, HID))
    P = {n: torch.zeros(s[n]) for n in ops.VARIANT_PARAMS[variant]}
    assert set(P) == set(s)
    return P


def _names(tensors, prefix=""):
    return {t.data_ptr(): prefix + n for n, t in tensors.items()}


def _describe(s, names):
    """field -> name of every non-NULL pointer field (array fields as field[i], NaisParams.branch[i].field) and every scalar field."""
    out = {}

    def put(key, typ, v):
        if typ.__name__ == "c_void_p":
            if v:
                out[key] = names[v]
        elif not key.startswith(("dropout", "pairs_precision", "dist_bucket_km", "reserved")):
            out[key] = round(v, 6) if isinstance(v, float) else v

    for f, typ in s._fields_:
        v = getattr(s, f)
        if f == "branch":
            for i in range(2):
                for bf, btyp in v[i]._fields_:
                    put(f"branch[{i}].{bf}", btyp, getattr(v[i], bf))
        elif hasattr(typ, "_length_"):
            for i in range(typ._length_):
                put(f"{f}[{i}]", typ._type_, v[i])
        else:
            put(f, typ, v)
    return out


@pytest.mark.parametrize("variant", list(EXPECTED))
def test_params_and_optimizer_state_slots(variant):
    P = _params(variant)
    keep = []
    p = ops.build_params(variant, P, 0.5, keep)
    assert _describe(p, _names(P)) == EXPECTED[variant]["params"]
    assert {t.data_ptr() for t in keep} == {t.data_ptr() for t in P.values()}  # contiguous float32: no copies, all kept
    sums = {n: torch.zeros_like(t) for n, t in P.items()}
    o = ops._adagrad_struct(variant, P, sums, 0.5, 0.25, tables=True)
    assert _describe(o, _names(sums)) == EXPECTED[variant]["adagrad"]
    d = ops._adagrad_struct(variant, P, sums, 0.125, 0.0625, tables=False)
    assert _describe(d, _names(sums)) == EXPECTED[variant]["dense_adagrad"]


@pytest.mark.parametrize("variant", list(EXPECTED))
def test_grads_slots(variant):
    P = _params(variant)
    G = {n: torch.zeros_like(t) for n, t in P.items()}
    names = _names(G)
    e = EXPECTED[variant]
    assert _describe(ops._grads_struct(variant, ops._addresses(G)), names) == e["grads_tables"]
    mlp = {n: t for n, t in G.items() if n not in ops._TABLES}
    assert _describe(ops._grads_struct(variant, ops._addresses(mlp)), names) == e["grads_no_tables"]
    if variant == "disentangled":  # (row-compacted gradients and the presorting forward: one-branch variants only)
        assert "grads_compact" not in e and "grads_presort" not in e
        return
    rows = {n: torch.zeros_like(G[n]) for n in ops._TABLES if n in P}
    remaps = {n: torch.zeros(P[n].shape[0], dtype=torch.int32) for n in rows}
    g = ops._grads_struct(variant, {**ops._addresses(mlp), **ops._addresses(rows)}, ops._addresses(remaps))
    assert _describe(g, {**names, **_names(rows, "rows:"), **_names(remaps, "remap:")}) == e["grads_compact"]
    ws = torch.zeros(16, dtype=torch.uint8)
    g = ops._grads_struct(variant, {n: ws.data_ptr() for n in ops.VARIANT_PARAMS[variant] if n in ops._TABLES})
    assert _describe(g, {ws.data_ptr(): "ws"}) == e["grads_presort"]


def test_derived_name_lists():
    assert ops._TABLES == ("embed_history.weight", "embed_target.weight", "embed_region.weight")
    assert ops._FULLY_WRITTEN == {"attn_layer1.weight", "attn_layer1.bias", "attn_layer2.weight", "dist_layer.weight", "dist_layer.bias",
                                  "region_attn_layer1.weight", "region_attn_layer1.bias", "region_attn_layer2.weight"}
    for variant, e in EXPECTED.items():  # VARIANT_PARAMS keeps the state_dict order
        assert set(ops.VARIANT_PARAMS[variant]) == set(_params(variant))
    assert ops.VARIANT_PARAMS["disentangled"] == (
        "embed_history.weight", "embed_target.weight", "embed_region.weight", "embed_distance.weight", "attn_layer1.weight",
        "attn_layer1.bias", "attn_layer2.weight", "region_attn_layer1.weight", "region_attn_layer1.bias", "region_attn_layer2.weight")


@pytest.mark.parametrize("variant", ["region", "disentangled"])
def test_wrong_optimizer_state_raises(variant):
    P = _params(variant)
    for name, tables in (("embed_region.weight", True), ("attn_layer1.weight", False)):
        for bad in (torch.zeros(3), torch.zeros_like(P[name], dtype=torch.float64), torch.zeros(P[name].shape[::-1]).t()):
            sums = {n: torch.zeros_like(t) for n, t in P.items()}
            sums[name] = bad
            with pytest.raises(RuntimeError, match=f"fused Adagrad: {name} and its state must be contiguous float32 of the same shape"):
                ops._adagrad_struct(variant, P, sums, 0.5, 0.25, tables)


def test_attention_layer_shape_is_checked():
    P = _params("region_distance")
    P["attn_layer1.weight"] = torch.zeros(HID, 8)  # the lat/lon lanes missing
    with pytest.raises(RuntimeError, match="attn_layer shapes do not match the variant"):
        ops.build_params("region_distance", P, 0.5, [])
