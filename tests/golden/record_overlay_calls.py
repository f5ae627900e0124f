"""Records how the UNMODIFIED reference drives the ptgnn_b200 classes once ``ptgnn_b200.overlay.install()`` is in place.

    python tests/golden/record_overlay_calls.py     # writes tests/golden/overlay_calls.json

Needs the reference tree (see ``oracle/refimport.py``).  Installs the overlay, then builds the Typilus Graph2Class model
with the reference's own factory (``create_graph2class_gnn_model``) and feeds it a tensorised minibatch, as a user of the
reference would.  It stores, in call order, every constructor call of a ptgnn_b200 class (class name, positional and keyword
arguments), the reference residual layers placed in the layer list, the keys of ``finalize_minibatch()`` and the keyword
arguments (by type) that reach ``GraphNeuralNetwork.forward``.  ``tests/test_overlay_cpu.py`` replays exactly these calls
through a stand-in package, so the check needs no reference tree.
"""
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.refimport import REFERENCE_ROOT, reference_available  # noqa: E402

if not reference_available():
    sys.exit(f"reference tree not found at {REFERENCE_ROOT}")
sys.path.insert(0, os.path.join(ROOT, "oracle", "refstubs"))
sys.path.insert(0, REFERENCE_ROOT)

import torch  # noqa: E402

import ptgnn_b200 as P  # noqa: E402
import ptgnn_b200.overlay as ov  # noqa: E402

ov.install(force_torch_scatter=True)       # before any reference import, as a user of the overlay does

HIDDEN = 64
calls, built, residuals, forward = [], {}, {}, {}


def encode(v):
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    if isinstance(v, (list, tuple)):
        return [encode(x) for x in v]
    if id(v) in built:
        return {"ref": built[id(v)]}
    name = type(v).__name__
    if name == "_ResidualOriginLayer":
        return {"residual_origin_of": encode(v._ResidualOriginLayer__target_layer)["residual"]}
    if name.endswith("ResidualLayer"):
        if id(v) not in residuals:
            residuals[id(v)] = (len(residuals), {"class": name, "input_dim": v.input_state_dimension})
        return {"residual": residuals[id(v)][0]}
    if isinstance(v, torch.nn.Module):
        return {"module": type(v).__module__ + "." + name}
    raise TypeError(f"cannot record a {type(v)}")


def describe(v):
    if torch.is_tensor(v):
        return {"tensor": str(v.dtype).replace("torch.", ""), "dim": v.dim()}
    if isinstance(v, dict):
        return {"dict": {k: describe(x) for k, x in v.items()}}
    if isinstance(v, (list, tuple)):
        return {"list": [describe(x) for x in v]}
    if v is None or isinstance(v, (bool, int, float, str)):
        return {"value": v}
    raise TypeError(f"cannot describe a {type(v)}")


def recording(cls):
    init = cls.__init__

    def __init__(self, *args, **kwargs):
        call = {"class": cls.__name__, "args": encode(args), "kwargs": {k: encode(x) for k, x in kwargs.items()}}
        init(self, *args, **kwargs)
        built[id(self)] = len(calls)
        calls.append(call)

    cls.__init__ = __init__


for cls in (P.GatedMessagePassingLayer, P.MlpMessagePassingLayer, P.GraphNeuralNetwork):
    recording(cls)
container_forward = P.GraphNeuralNetwork.forward


def recording_forward(self, **kwargs):
    forward.update({k: describe(x) for k, x in kwargs.items()})
    return container_forward(self, **kwargs)


P.GraphNeuralNetwork.forward = recording_forward

import ptgnn.implementations.typilus.train as typilus_train  # noqa: E402

random.seed(0)


def sample():
    n = 12
    nodes = [random.choice(["foo_bar", "baz", "x", "getValue", "int", "self"]) for _ in range(n)]
    edges = {"NEXT": {str(j): [j + 1] for j in range(n - 1)}, "CHILD": {"0": [3, 4], "5": [6]}, "OCCURRENCE_OF": {}}
    return {"nodes": nodes, "edges": edges, "token-sequence": list(range(n)),
            "supernodes": {"2": {"name": "a", "annotation": random.choice(["int", "str"])}, "7": {"name": "b", "annotation": "int"}}}


data = [sample() for _ in range(8)]
model = typilus_train.create_graph2class_gnn_model(hidden_state_size=HIDDEN)
model.compute_metadata(iter(data), parallelize=False)
nn_module = model.build_neural_module()
mb = model.initialize_minibatch()
for d in data[:3]:
    model.extend_minibatch_with(model.tensorize(d), mb)
final = model.finalize_minibatch(mb, "cpu")
try:
    with torch.no_grad():
        nn_module.eval()(**final)
except P._native.NativeLibraryError:       # the first ptgnn_b200 layer refuses CPU tensors: the inputs got that far
    pass
assert forward, "the minibatch never reached GraphNeuralNetwork.forward"
out = {
    "factory": {"name": "create_graph2class_gnn_model", "kwargs": {"hidden_state_size": HIDDEN}},
    "calls": calls,
    "residuals": [r for _, r in sorted(residuals.values(), key=lambda r: r[0])],
    "minibatch_keys": sorted(final),
    "graph_mb_data_keys": sorted(final["graph_mb_data"]) if "graph_mb_data" in final else None,
    "forward": forward,
}
path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "overlay_calls.json")
with open(path, "w") as f:
    json.dump(out, f, indent=1)
    f.write("\n")
print(path, len(calls), "calls")
