"""`ptgnn_b200.overlay.install()`: the reference's own packages build ptgnn_b200 layers WITHOUT being edited.

The reference is not part of this repository, so the test replays what the reference does instead of importing it.
``tests/golden/overlay_calls.json`` (written by ``tests/golden/record_overlay_calls.py`` from the unmodified reference) holds
every constructor call the reference's Typilus factory and ``GraphNeuralNetworkModel.build_neural_module`` make on the
ptgnn_b200 classes (class, positional and keyword arguments, in order), the residual layers it places in the layer list, and
the minibatch that reaches ``GraphNeuralNetwork.forward``.  The test writes a stand-in package with the reference's module
paths and import patterns into a temporary directory; its factory replays exactly those recorded calls.  Its own layer and
container classes raise when constructed, so a class the overlay fails to replace fails the test, and so does a ptgnn_b200
constructor or forward that no longer accepts what the reference passes.  Runs in a fresh interpreter because the point is
import order: overlay first, then ``ptgnn.implementations.*``."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORDED_CALLS = os.path.join(ROOT, "tests", "golden", "overlay_calls.json")

_STANDIN_CLASS = '''
from torch import nn


class {name}(nn.Module):
    def __init__(self, *args, **kwargs):
        raise AssertionError("stand-in {name} constructed: the overlay did not replace it")
'''

STANDIN_PACKAGE = {
    "ptgnn/__init__.py": "",
    "ptgnn/_replay.py": '''
        import torch
        from torch import nn


        class NodeEmbedder(nn.Module):
            """Takes the place of the reference's node embedder: one zero row of width `width` per node."""

            def __init__(self, width):
                super().__init__()
                self.width = width

            def forward(self, **node_data):
                n = next(t for t in node_data.values() if torch.is_tensor(t)).shape[0]
                return torch.zeros(n, self.width)


        class Replay:
            """Makes the recorded constructor calls.  An argument {"ref": i} is the object made by recorded call i,
            {"residual": j} the package's residual layer j, {"residual_origin_of": j} a pass-through origin of it and
            {"module": name} a stand-in node embedder."""

            def __init__(self, recorded, hidden_state_size):
                self.recorded, self.hidden = recorded, hidden_state_size
                self.built, self.residuals = [], {}

            def residual(self, j):
                if j not in self.residuals:
                    from ptgnn.neuralmodels.gnn.messagepassing import residuallayers

                    spec = self.recorded["residuals"][j]
                    self.residuals[j] = getattr(residuallayers, spec["class"])(spec["input_dim"])
                return self.residuals[j]

            def value(self, v):
                if isinstance(v, list):
                    return [self.value(x) for x in v]
                if not isinstance(v, dict):
                    return v
                if "ref" in v:
                    return self.built[v["ref"]]
                if "residual" in v:
                    return self.residual(v["residual"])
                if "residual_origin_of" in v:
                    return self.residual(v["residual_origin_of"]).pass_through_dummy_layer()
                return NodeEmbedder(self.hidden)

            def call(self, cls, call):
                assert cls.__name__ == call["class"], (cls, call["class"])
                obj = cls(*self.value(call["args"]), **{k: self.value(x) for k, x in call["kwargs"].items()})
                self.built.append(obj)
                return obj
    ''',
    "ptgnn/baseneuralmodel/__init__.py": "from .modulewithmetrics import ModuleWithMetrics\n",
    "ptgnn/baseneuralmodel/modulewithmetrics.py": '''
        from abc import ABC

        from torch import nn


        class ModuleWithMetrics(nn.Module, ABC):
            """Only the name and the ABC matter here: the overlay registers the ptgnn_b200 container with this class."""
    ''',
    "ptgnn/neuralmodels/__init__.py": "",
    "ptgnn/neuralmodels/gnn/__init__.py": "from .graphneuralnetwork import GraphNeuralNetwork, GraphNeuralNetworkModel\n",
    "ptgnn/neuralmodels/gnn/graphneuralnetwork.py": '''
        from ptgnn.baseneuralmodel import ModuleWithMetrics


        class GraphNeuralNetwork(ModuleWithMetrics):
            def __init__(self, *args, **kwargs):
                raise AssertionError("stand-in GraphNeuralNetwork constructed: the overlay did not replace it")


        class GraphNeuralNetworkModel:
            def __init__(self, replay, message_passing_layer_creator):
                self.__replay = replay
                self.__create_layers = message_passing_layer_creator

            def build_neural_module(self):
                self.__create_layers()
                return self.__replay.call(GraphNeuralNetwork, self.__replay.recorded["calls"][-1])   # looked up at call time
    ''',
    "ptgnn/neuralmodels/gnn/messagepassing/__init__.py": '''
        from .abstractmessagepassing import AbstractMessagePassingLayer
        from .gatedmessagepassing import GatedMessagePassingLayer
        from .mlpmessagepassing import MlpMessagePassingLayer
        from .residuallayers import ConcatResidualLayer
    ''',
    "ptgnn/neuralmodels/gnn/messagepassing/abstractmessagepassing.py":
        _STANDIN_CLASS.format(name="AbstractMessagePassingLayer") + _STANDIN_CLASS.format(name="AbstractMessageAggregation"),
    "ptgnn/neuralmodels/gnn/messagepassing/gatedmessagepassing.py": _STANDIN_CLASS.format(name="GatedMessagePassingLayer"),
    "ptgnn/neuralmodels/gnn/messagepassing/mlpmessagepassing.py": _STANDIN_CLASS.format(name="MlpMessagePassingLayer"),
    "ptgnn/neuralmodels/gnn/messagepassing/residuallayers.py": '''
        import torch

        from ptgnn.neuralmodels.gnn.messagepassing.abstractmessagepassing import AbstractMessagePassingLayer


        class _PassThrough(AbstractMessagePassingLayer):
            """Hands its input states to a residual layer further down the stack and returns them unchanged."""

            def __init__(self, residual):
                super().__init__()
                self.__residual = [residual]

            def forward(self, node_states, **unused):
                self.__residual[0].saved_states = node_states
                return node_states


        class ConcatResidualLayer(AbstractMessagePassingLayer):
            """Appends the states saved by its pass-through origin to its input states."""

            def __init__(self, input_dim):
                super().__init__()
                self.saved_states = None
                self.__input_dim = input_dim

            def pass_through_dummy_layer(self):
                return _PassThrough(self)

            def forward(self, node_states, **unused):
                return torch.cat([self.saved_states, node_states], dim=-1)

            @property
            def input_state_dimension(self):
                return self.__input_dim

            @property
            def output_state_dimension(self):
                return 2 * self.__input_dim
    ''',
    "ptgnn/implementations/__init__.py": "",
    "ptgnn/implementations/typilus/__init__.py": "",
    "ptgnn/implementations/typilus/train.py": '''
        from ptgnn._replay import Replay
        from ptgnn.baseneuralmodel import ModuleWithMetrics
        from ptgnn.neuralmodels.gnn import GraphNeuralNetworkModel
        from ptgnn.neuralmodels.gnn.messagepassing import GatedMessagePassingLayer, MlpMessagePassingLayer

        LAYER_CLASSES = {"GatedMessagePassingLayer": GatedMessagePassingLayer, "MlpMessagePassingLayer": MlpMessagePassingLayer}


        def create_graph2class_gnn_model(recorded, hidden_state_size):
            replay = Replay(recorded, hidden_state_size)

            def create_layers():
                for call in recorded["calls"][:-1]:
                    replay.call(LAYER_CLASSES[call["class"]], call)

            return GraphNeuralNetworkModel(replay, create_layers)


        class Graph2ClassModule(ModuleWithMetrics):
            def __init__(self, gnn):
                super().__init__()
                self.gnn = gnn
                self.num_samples = 0

            def _module_metrics(self):
                return {"num_samples": self.num_samples}

            def _reset_module_metrics(self):
                self.num_samples = 0

            def forward(self, graph_mb_data, **targets):
                return self.gnn(**graph_mb_data)
    ''',
    "ptgnn/implementations/graph2seq/__init__.py": "",
    "ptgnn/implementations/graph2seq/train.py": '''
        from ptgnn.neuralmodels.gnn.graphneuralnetwork import GraphNeuralNetworkModel
        from ptgnn.neuralmodels.gnn.messagepassing.gatedmessagepassing import GatedMessagePassingLayer
    ''',
}

SCRIPT = r'''
import inspect, json, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {standin!r})
with open({recorded!r}) as f:
    recorded = json.load(f)
import ptgnn_b200 as P
import ptgnn_b200.overlay as ov
report = ov.install(force_torch_scatter=True)
assert report["layers"] and report["container"] and report["metrics"], report
import torch_scatter
assert torch_scatter.__name__ == "ptgnn_b200.torch_scatter_shim" and hasattr(torch_scatter, "scatter_log_softmax")
from torch_scatter.composite import scatter_logsumexp      # the form the reference's decoder imports

# --- the package's factories, imported AFTER the overlay, unchanged ---
import ptgnn.implementations.typilus.train as typilus_train
import ptgnn.implementations.graph2seq.train as g2s_train   # imports GatedMessagePassingLayer by module path
from ptgnn.baseneuralmodel import ModuleWithMetrics
import ptgnn.neuralmodels.gnn as ref_gnn_pkg
import ptgnn.neuralmodels.gnn.graphneuralnetwork as ref_gnn_mod
assert typilus_train.GatedMessagePassingLayer is P.GatedMessagePassingLayer
assert typilus_train.MlpMessagePassingLayer is P.MlpMessagePassingLayer
assert g2s_train.GatedMessagePassingLayer is P.GatedMessagePassingLayer
assert ref_gnn_mod.GraphNeuralNetwork is P.GraphNeuralNetwork and ref_gnn_pkg.GraphNeuralNetwork is P.GraphNeuralNetwork
from ptgnn.neuralmodels.gnn.messagepassing.residuallayers import ConcatResidualLayer as RefConcat
assert issubclass(RefConcat, P.AbstractMessagePassingLayer)     # the package's residual layers now derive from our base

# --- the reference's constructor calls, replayed through the package's factory ---
model = typilus_train.create_graph2class_gnn_model(recorded, **recorded["factory"]["kwargs"])
gnn = model.build_neural_module()
assert type(gnn) is P.GraphNeuralNetwork, "the package built our container"
layers = list(gnn.message_passing_layers)
kinds = [type(l).__module__ + "." + type(l).__name__ for l in layers]
assert len(layers) == 12, kinds
assert kinds.count("ptgnn_b200.messagepassing.MlpMessagePassingLayer") == 8, kinds
assert [l.input_state_dimension for l in layers if isinstance(l, P.MlpMessagePassingLayer)].count(128) == 2, kinds
assert kinds.count("ptgnn.neuralmodels.gnn.messagepassing.residuallayers.ConcatResidualLayer") == 2, kinds
assert kinds.count("ptgnn.neuralmodels.gnn.messagepassing.residuallayers._PassThrough") == 2, kinds
# --- metrics protocol: a parent of the package finds our container among its ModuleWithMetrics children ---
assert isinstance(gnn, ModuleWithMetrics)
nn_module = typilus_train.Graph2ClassModule(gnn)
gnn._GraphNeuralNetwork__num_edges = 7; gnn._GraphNeuralNetwork__num_nodes = 3; gnn._GraphNeuralNetwork__num_graphs = 1
nn_module.num_samples = 1
children = [m for m in nn_module.modules() if isinstance(m, ModuleWithMetrics)]
assert gnn in children
metrics = {{k: v for m in children for k, v in m._module_metrics().items()}}
assert metrics == {{"num_samples": 1, "num_graphs": 1, "num_nodes": 3, "num_edges": 7}}, metrics
for m in children:
    m._reset_module_metrics()
assert gnn._module_metrics() == {{"num_graphs": 0, "num_nodes": 0, "num_edges": 0}}
# --- the reference's minibatch reaches the container's forward (CPU: no kernel call) ---
import torch
forward = recorded["forward"]
assert sorted(forward) == recorded["graph_mb_data_keys"], "GraphNeuralNetwork.forward receives finalize_minibatch()['graph_mb_data']"
accepted = {{n for n, p in inspect.signature(P.GraphNeuralNetwork.forward).parameters.items() if p.kind is p.KEYWORD_ONLY}}
assert set(forward) <= accepted, sorted(set(forward) - accepted)

def rebuild(d, n=5):
    if "tensor" in d:
        return torch.zeros((n,) + (3,) * (d["dim"] - 1), dtype=getattr(torch, d["tensor"]))
    if "dict" in d:
        return {{k: rebuild(v) for k, v in d["dict"].items()}}
    if "list" in d:
        return [rebuild(v) for v in d["list"]]
    return d["value"]

final = {{k: None for k in recorded["minibatch_keys"]}}
final["graph_mb_data"] = {{k: rebuild(v) for k, v in forward.items()}}
try:
    with torch.no_grad():
        nn_module.eval()(**final)
except P._native.NativeLibraryError as e:      # reaches the first ptgnn_b200 layer, which refuses CPU tensors (no fallback)
    assert "no CPU fallback" in str(e)
else:
    raise AssertionError("expected the ptgnn_b200 layer to refuse CPU tensors")
ov.uninstall()
assert ref_gnn_mod.GraphNeuralNetwork is not P.GraphNeuralNetwork
print("OVERLAY-OK", kinds[:3])
'''


def test_reference_implementations_build_ptgnn_b200_layers_unchanged(tmp_path):
    standin = tmp_path / "standin"
    for rel, src in STANDIN_PACKAGE.items():
        path = standin / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(textwrap.dedent(src).lstrip())
    code = SCRIPT.format(root=ROOT, standin=str(standin), recorded=RECORDED_CALLS)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode == 0 and "OVERLAY-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_overlay_without_reference_installs_only_the_shim(tmp_path):
    code = ("import sys; sys.path.insert(0, %r)\nimport ptgnn_b200.overlay as ov\nr = ov.install(force_torch_scatter=True)\n"
            "import torch_scatter\nassert torch_scatter.__name__ == 'ptgnn_b200.torch_scatter_shim'\n"
            "assert r['layers'] is False and 'note' in r, r\nprint('SHIM-OK')\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert r.returncode == 0 and "SHIM-OK" in r.stdout, r.stdout + r.stderr[-3000:]
