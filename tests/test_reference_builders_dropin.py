"""CPU: "drop-in", literally.

The SOURCE FILES of the reference's five builders (deepctr/models/{deepfm,xdeepfm,dcn,autoint}.py,
deepctr/models/sequence/din.py), executed unmodified with their imports aliased to this package
(tests/golden/generate_builders.py), built the graphs stored in tests/golden/reference_builders.json.

The graphs deepctr_b200.models builds for the same columns must be those: same inputs, same layer
sequence (class + Keras-style name), same weights (name + shape + trainable), same planner slots (i.e.
the same single fused gather launch).  Graph construction needs no GPU.
"""
import inspect
import json
import os

import pytest

import golden_models as G

with open(os.path.join(os.path.dirname(G.MODELS), "reference_builders.json")) as _f:
    REF = json.load(_f)
BUILDERS = ("DeepFM", "xDeepFM", "DCN", "AutoInt", "DIN")


@pytest.mark.parametrize("name", G.CASES)
def test_reference_builder_source_runs_on_this_package(name):
    fx = G.Fixture(name)
    a = REF["graphs"][name]
    b = json.loads(json.dumps(G.graph_signature(G.build_model(fx))))
    assert a["inputs"] == b["inputs"]
    assert a["weights"] == b["weights"]
    assert a["slots"] == b["slots"] and a["fast"] == b["fast"]
    # the op graph: same multiset of (layer class, name); the topological order may differ where the
    # reference builds a branch earlier than it consumes it
    assert sorted(a["layers"]) == sorted(b["layers"])


def test_reference_default_arguments_are_the_same():
    """every keyword and default of the five reference builders exists here with the same default."""
    from deepctr_b200 import models as M
    assert sorted(REF["defaults"]) == sorted(BUILDERS)
    for name in BUILDERS:
        mine = [[k, repr(p.default)] for k, p in inspect.signature(getattr(M, name)).parameters.items()]
        assert [k for k, _ in REF["defaults"][name]] == [k for k, _ in mine], name
        assert REF["defaults"][name] == mine, name
