"""Shared loader for the MODEL-level golden fixtures (tests/golden/models/*.npz, produced by the
reference's own feature_column.py / inputs.py / builders under the TF shim: see
tests/golden/generate_models.py) and the two mappings a test needs:

* ``oracle_weights``  fixture weight keys -> the dict oracle/models.py takes;
* ``assign_weights``  fixture weight keys -> the weights of a deepctr_b200 model built from the same columns.

Key convention of the fixtures: ``<top-level layer name>/<reference attribute path>/<weight name>``.
``linearsparse_emb_*`` tables are the reference's redundant second lookup pass inside get_linear_logit
(feature_column.py:185, SURVEY.md App. F.2): their outputs are discarded, their gradient is zero, and
neither the oracle nor this package materialises them.
"""
import glob
import json
import os

import numpy as np
import torch

MODELS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models")
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(MODELS, "*.npz")))


class Fixture(object):
    def __init__(self, name):
        d = np.load(os.path.join(MODELS, name + ".npz"))
        self.name = name
        self.meta = json.loads(str(d["meta"]))
        self.x = {k[2:]: d[k] for k in d.files if k.startswith("x_")}
        self.y = d["y"]
        self.w = {k[2:]: d[k] for k in d.files if k.startswith("w_")}
        self.g = {k[2:]: d[k] for k in d.files if k.startswith("g_")}
        self.out, self.logit, self.loss = d["out"], d["logit"], float(d["loss"])
        self.builder, self.kwargs = self.meta["builder"], self.meta["kwargs"]
        self.task = self.meta.get("task", "binary")
        self.training = bool(self.meta.get("training"))

    def layer_names(self, cls):
        return [n for c, n in self.meta["layers"] if c == cls]

    def inputs(self):
        """what a user passes: ints as int32/int64 arrays, strings as str arrays, floats as float32."""
        out = {}
        for k, a in self.x.items():
            out[k] = a.astype(np.int32) if a.dtype.kind in "iu" else a
        return out


def columns(fx, which, FC):
    """Rebuild the feature columns with module ``FC``'s SparseFeat / VarLenSparseFeat / DenseFeat."""
    def sparse(m):
        vp = os.path.join(MODELS, m["vocabulary_path"]) if m["vocabulary_path"] else None
        return FC.SparseFeat(m["name"], m["vocabulary_size"], m["embedding_dim"], use_hash=m["use_hash"],
                             vocabulary_path=vp, dtype=m["dtype"], embedding_name=m["embedding_name"],
                             group_name=m["group_name"], trainable=m["trainable"])
    out = []
    for m in fx.meta["columns"][which]:
        if m["kind"] == "sparse":
            out.append(sparse(m))
        elif m["kind"] == "varlen":
            out.append(FC.VarLenSparseFeat(sparse(m["sparsefeat"]), maxlen=m["maxlen"], combiner=m["combiner"],
                                           length_name=m["length_name"], weight_name=m["weight_name"],
                                           weight_norm=m["weight_norm"]))
        else:
            out.append(FC.DenseFeat(m["name"], m["dimension"]))
    return out


def _ignored(key):
    return key.startswith("linearsparse_")


def oracle_weights(fx, requires_grad=False):
    """-> (W for oracle/models.py, {fixture key: leaf tensor})."""
    leaves = {}

    def t(key):
        v = torch.tensor(fx.w[key], requires_grad=requires_grad and key in fx.g)
        leaves[key] = v
        return v

    W = {"tables": {}, "att": []}
    for name in fx.layer_names("Embedding"):
        if not _ignored(name):
            W["tables"][name] = t(name + "/embeddings")
    for name in fx.layer_names("DNN"):
        n = len([k for k in fx.w if k.startswith(name + "/kernel")])
        W["dnn_kernels"] = [t("%s/kernel%d" % (name, i)) for i in range(n)]
        W["dnn_biases"] = [t("%s/bias%d" % (name, i)) for i in range(n)]
    for name in fx.layer_names("Linear"):
        if name + "/linear_kernel" in fx.w:
            W["linear_kernel"] = t(name + "/linear_kernel")
    denses = fx.layer_names("Dense")
    if denses:
        W["dense_kernel"] = t(denses[0] + "/kernel")
    if len(denses) > 1:
        W["cin_dense_kernel"] = t(denses[1] + "/kernel")
    for name in fx.layer_names("PredictionLayer"):
        if name + "/global_bias" in fx.w:
            W["global_bias"] = t(name + "/global_bias")
    for name in fx.layer_names("CIN"):
        n = len([k for k in fx.w if k.startswith(name + "/filter")])
        W["cin_filters"] = [t("%s/filter%d" % (name, i)) for i in range(n)]
        W["cin_biases"] = [t("%s/bias%d" % (name, i)) for i in range(n)]
    for name in fx.layer_names("CrossNet"):
        n = len([k for k in fx.w if k.startswith(name + "/kernel")])
        W["cross_kernels"] = [t("%s/kernel%d" % (name, i)) for i in range(n)]
        W["cross_biases"] = [t("%s/bias%d" % (name, i)) for i in range(n)]
    for name in fx.layer_names("InteractingLayer"):
        d = {"query": t(name + "/query"), "key": t(name + "/key"), "value": t(name + "/value")}
        if name + "/res" in fx.w:
            d["res"] = t(name + "/res")
        W["att"].append(d)
    for name in fx.layer_names("AttentionSequencePoolingLayer"):
        p = name + "/local_att/"
        n = len([k for k in fx.w if k.startswith(p + "dnn/kernel")])
        d = {"dnn_kernels": [t("%sdnn/kernel%d" % (p, i)) for i in range(n)],
             "dnn_biases": [t("%sdnn/bias%d" % (p, i)) for i in range(n)],
             "kernel": t(p + "kernel"), "bias": t(p + "bias")}
        acts = []
        for i in range(n):
            a = "%sdnn/activation_layers%d/" % (p, i)
            if a + "dice_alpha" in fx.w:
                acts.append({"alphas": t(a + "dice_alpha"), "moving_mean": t(a + "bn/moving_mean"),
                             "moving_var": t(a + "bn/moving_variance")})
            else:
                acts.append(None)
        if any(a is not None for a in acts):
            d["act_params"] = acts
        W["lau"] = d
    return W, leaves


def oracle_forward(fx, W, FC):
    """(logit, prediction) of oracle/models.py for this fixture's builder + kwargs."""
    from oracle import models as OM
    kw = fx.kwargs
    x = fx.inputs()
    lin, dnn = columns(fx, "linear", FC), columns(fx, "dnn", FC)
    b = fx.builder
    if b == "DeepFM":
        return OM.deepfm(x, lin, dnn, W, fm_group=tuple(kw.get("fm_group", ("default_group",))), task=fx.task)
    if b == "xDeepFM":
        return OM.xdeepfm(x, lin, dnn, W, cin_layer_size=tuple(kw["cin_layer_size"]),
                          cin_split_half=kw["cin_split_half"], cin_activation=kw["cin_activation"], task=fx.task)
    if b == "DCN":
        return OM.dcn(x, lin, dnn, W, cross_num=kw["cross_num"], parameterization=kw["cross_parameterization"],
                      use_dnn=len(kw["dnn_hidden_units"]) > 0, task=fx.task)
    if b == "AutoInt":
        return OM.autoint(x, lin, dnn, W, att_layer_num=kw["att_layer_num"],
                          att_embedding_size=kw["att_embedding_size"], att_head_num=kw["att_head_num"],
                          att_res=kw["att_res"], use_dnn=len(kw["dnn_hidden_units"]) > 0, task=fx.task)
    if b == "DIN":
        return OM.din(x, dnn, ["item_id", "cate_id"], W, att_activation=kw["att_activation"],
                      att_weight_normalization=kw["att_weight_normalization"], task=fx.task,
                      training=fx.training)
    raise KeyError(b)


def loss_of(fx, pred):
    """Keras binary_crossentropy on probabilities / mse (SURVEY.md App. C)."""
    from oracle import ops as O
    if fx.task == "binary":
        return O.binary_crossentropy(fx.y, pred)
    y = torch.as_tensor(fx.y).reshape(-1, 1)
    return ((pred - y) ** 2).mean()


# ---- deepctr_b200 side -------------------------------------------------------------------------------
_RENAMES = [("/local_att/", "/local_activation_unit/"), ("/activation_layers", "/act")]


def build_model(fx):
    """Build the deepctr_b200 model of this fixture (graph construction only: works without a GPU)."""
    from deepctr_b200 import engine as E
    from deepctr_b200 import feature_column as FC
    from deepctr_b200 import models as M
    E.clear_session()
    kw = dict(fx.kwargs)
    for k in ("dnn_hidden_units", "cin_layer_size", "att_hidden_size", "fm_group"):
        if k in kw:
            kw[k] = tuple(kw[k])
    lin, dnn = columns(fx, "linear", FC), columns(fx, "dnn", FC)
    if fx.builder == "DIN":
        return M.DIN(dnn, ["item_id", "cate_id"], **kw)
    return getattr(M, fx.builder)(lin, dnn, **kw)


def graph_signature(model):
    """What identifies a built graph: inputs, layers (class + Keras-style name), weights (name + shape +
    trainable) and the embedding planner's slots - plain lists, comparable with their JSON form."""
    from deepctr_b200 import engine as E
    layers = [[type(l).__name__, l.name] for l in model.layers if not isinstance(l, E.InputLayer)]
    weights = [[w.name, list(w.shape), w.trainable] for w in model.weights]
    slots = [[s.emb.name, s.input_name, s.maxlen, s.pool, s.mask_mode, s.len_name, s.weight_name, s.weight_mode,
              s.dim, s.buf, s.col] for s in model.planner.slots]
    return {"inputs": list(model.input_names), "layers": layers, "weights": weights, "slots": slots,
            "fast": [model.planner.fast, getattr(model.planner, "fast_n", 0)]}


def weight_map(fx, model):
    """{fixture key: deepctr_b200 Weight}; raises if the two weight sets differ (names or shapes)."""
    mine = {w.name: w for w in model.weights}
    out, missing = {}, []
    for key, val in fx.w.items():
        if _ignored(key):
            continue
        k2 = key
        for a, b in _RENAMES:
            k2 = k2.replace(a, b)
        if k2 not in mine:
            missing.append((key, k2))
            continue
        if tuple(mine[k2].shape) != tuple(val.shape):
            raise AssertionError("shape of %s: reference %s, here %s" % (key, val.shape, mine[k2].shape))
        out[key] = mine.pop(k2)
    if missing or mine:
        raise AssertionError("weight sets differ: reference-only %s, here-only %s" % (missing, sorted(mine)))
    return out


def assign_weights(fx, model):
    wm = weight_map(fx, model)
    for key, w in wm.items():
        w.set_value(fx.w[key])
    return wm
