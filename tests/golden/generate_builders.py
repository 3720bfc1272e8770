#!/usr/bin/env python
"""Generate tests/golden/reference_builders.json: the graphs the REFERENCE's five builders build on this
package, and the builders' parameters with their defaults.

    python tests/golden/generate_builders.py <reference checkout>

The SOURCE FILES of the builders (deepctr/models/{deepfm,xdeepfm,dcn,autoint}.py,
deepctr/models/sequence/din.py) are executed unmodified with their imports aliased to this package:

    ..feature_column / ..inputs / ..layers.*      ->  deepctr_b200.feature_column / inputs / layers.*
    tensorflow.keras.models.Model, .layers.{Dense,Flatten,Concatenate}  ->  deepctr_b200.engine

For every model fixture under tests/golden/models/ the file holds golden_models.graph_signature() of the
graph the reference builder made from the fixture's columns and arguments; for every builder, each
parameter name with the repr() of its default.  Graph construction needs no GPU.
"""
import importlib.util
import inspect
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_builders.json")

import golden_models as G  # noqa: E402

FILES = {"DeepFM": ("models/deepfm.py", "models.deepfm"), "xDeepFM": ("models/xdeepfm.py", "models.xdeepfm"),
         "DCN": ("models/dcn.py", "models.dcn"), "AutoInt": ("models/autoint.py", "models.autoint"),
         "DIN": ("models/sequence/din.py", "models.sequence.din")}


class _aliased(object):
    """sys.modules entries that make the reference builder files import this package; restored on exit."""

    def __enter__(self):
        import deepctr_b200  # noqa: F401
        from deepctr_b200 import engine, feature_column, inputs, layers
        from deepctr_b200.layers import core, interaction, sequence, utils
        self.saved = {k: v for k, v in sys.modules.items() if k == "tensorflow" or k.startswith("tensorflow.")
                      or k == "refdrop" or k.startswith("refdrop.")}
        for k in self.saved:
            del sys.modules[k]

        def mod(name, **attrs):
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            m.__path__ = []
            sys.modules[name] = m
            return m
        tf = mod("tensorflow")
        tf.keras = mod("tensorflow.keras")
        tf.keras.models = mod("tensorflow.keras.models", Model=engine.Model)
        tf.keras.layers = mod("tensorflow.keras.layers", Dense=engine.Dense, Flatten=engine.Flatten,
                              Concatenate=engine.Concatenate)
        mod("refdrop")
        mod("refdrop.models")
        mod("refdrop.models.sequence")
        sys.modules["refdrop.feature_column"] = feature_column
        sys.modules["refdrop.inputs"] = inputs
        sys.modules["refdrop.layers"] = layers
        sys.modules["refdrop.layers.core"] = core
        sys.modules["refdrop.layers.interaction"] = interaction
        sys.modules["refdrop.layers.sequence"] = sequence
        sys.modules["refdrop.layers.utils"] = utils
        self.added = [k for k in sys.modules if k == "tensorflow" or k.startswith("tensorflow.")
                      or k == "refdrop" or k.startswith("refdrop.")]
        return self

    def __exit__(self, *a):
        for k in self.added:
            sys.modules.pop(k, None)
        sys.modules.update(self.saved)


def reference_builder(ref, name):
    rel, modname = FILES[name]
    full = "refdrop." + modname
    spec = importlib.util.spec_from_file_location(full, os.path.join(ref, "deepctr", rel))
    m = importlib.util.module_from_spec(spec)
    sys.modules[full] = m
    spec.loader.exec_module(m)            # the reference's unmodified source
    return getattr(m, name)


def builder_args(fx):
    from deepctr_b200 import feature_column as FC
    kw = dict(fx.kwargs)
    for k in ("dnn_hidden_units", "cin_layer_size", "att_hidden_size", "fm_group"):
        if k in kw:
            kw[k] = tuple(kw[k])
    lin, dnn = G.columns(fx, "linear", FC), G.columns(fx, "dnn", FC)
    if fx.builder == "DIN":
        return (dnn, ["item_id", "cate_id"]), kw
    return (lin, dnn), kw


def main(ref):
    from deepctr_b200 import engine as E
    out = {"graphs": {}, "defaults": {}}
    with _aliased():
        for name in G.CASES:
            fx = G.Fixture(name)
            args, kw = builder_args(fx)
            build = reference_builder(ref, fx.builder)
            E.clear_session()
            model = build(*args, **kw)
            G.weight_map(fx, model)       # the reference-built graph carries the fixture's weights by name
            out["graphs"][name] = G.graph_signature(model)
        for name in FILES:
            params = inspect.signature(reference_builder(ref, name)).parameters
            out["defaults"][name] = [[k, repr(p.default)] for k, p in params.items()]
    E.clear_session()
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("%s: %d graphs, %d builders" % (OUT, len(out["graphs"]), len(out["defaults"])))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
