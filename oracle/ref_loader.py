"""Import the UNMODIFIED reference modules (kaddly/GraphNeuralNetwork): from the checkout $GNN_REFERENCE_ROOT
names, else from the verbatim snapshot in the git-ignored oracle/_ref/ (tools/make_ref_snapshot.py).  The
reference is not part of this repository; without either, `available()` is False.

Used by tests/test_oracle_vs_reference_live.py and tests/golden/make_golden.py to pin the oracle
restatement, by tests/test_reference_substitution_gpu.py (the reference's own models / loops with the
drop-in layers substituted) and by bench.py's `--impl reference` arm.  Test / baseline infrastructure:
the product package never imports it.  The reference folders reuse top-level module names (`models`,
`data_utils`, `utils`, ...) so each folder is imported in isolation (SURVEY.md §8c shims).
"""
import contextlib
import importlib
import importlib.util
import os
import sys
import warnings

_SNAPSHOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")

REF_ROOT = os.environ.get("GNN_REFERENCE_ROOT") or _SNAPSHOT
_SHARED_NAMES = ("models", "data_utils", "sample_utils", "graph_utils", "utils", "train_utils", "train_eval",
                 "GCN", "GraphSAGE")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "GCN"))


def _purge():
    for name in list(sys.modules):
        if name.split(".")[0] in _SHARED_NAMES:
            del sys.modules[name]


@contextlib.contextmanager
def folder(name):
    """sys.path / sys.modules isolated view of one reference folder."""
    path = os.path.join(REF_ROOT, name)
    _purge()
    sys.path.insert(0, path)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            yield path
    finally:
        sys.path.remove(path)
        _purge()


def load_file(relpath, modname):
    spec = importlib.util.spec_from_file_location(modname, os.path.join(REF_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def gcn():
    """(GCN.py module, data_utils module) of the GCN folder."""
    with folder("GCN"):
        return load_file("GCN/GCN.py", "ref_gcn_GCN"), load_file("GCN/data_utils.py", "ref_gcn_data_utils")


def gat_layers():
    """GAT/models/layers.py (GraphAttentionLayer, SpGraphAttentionLayer, SpecialSpmmFunction)."""
    return load_file("GAT/models/layers.py", "ref_gat_layers")


def gat_models():
    """GAT/models/GAT.py; its `from models.HAN import ...` (GAT/models/GAT.py:4) names a module
    that does not exist in the GAT folder — shimmed to GAT/models/layers.py (SURVEY.md §8c)."""
    layers = gat_layers()
    with folder("GAT"):
        pkg = type(sys)("models")
        pkg.__path__ = []
        sys.modules["models"] = pkg
        sys.modules["models.HAN"] = layers
        return load_file("GAT/models/GAT.py", "ref_gat_GAT"), layers


def sage_pytorch():
    """GraphSAGE_Pytorch: (models package, sample_utils module)."""
    with folder("GraphSAGE_Pytorch"):
        models = importlib.import_module("models")
        agg = importlib.import_module("models.Aggregator")
        sg = importlib.import_module("models.SageGCN")
        gs = importlib.import_module("models.GraphSage")
        su = importlib.import_module("sample_utils")
        return {"Aggregator": agg, "SageGCN": sg, "GraphSage": gs, "sample_utils": su, "models": models}


def sage_v2():
    """GraphSAGE (dedup variant): graph_utils, GraphSAGE, data_utils."""
    with folder("GraphSAGE"):
        gu = importlib.import_module("graph_utils")
        m = importlib.import_module("GraphSAGE")
        du = importlib.import_module("data_utils")
        return {"graph_utils": gu, "GraphSAGE": m, "data_utils": du}


def han():
    """HAN/models package (NodeAttention, SemanticAttention, HAN)."""
    with folder("HAN"):
        na = importlib.import_module("models.NodeAttention")
        sa = importlib.import_module("models.SemanticAttention")
        hm = importlib.import_module("models.HAN")
        return {"NodeAttention": na, "SemanticAttention": sa, "HAN": hm}


def gatne():
    """(GATNE_Pytorch/models/GATNE.py, GATNE/models/GATNE.py) — both files import torch only."""
    return load_file("GATNE_Pytorch/models/GATNE.py", "ref_gatne_pytorch"), load_file("GATNE/models/GATNE.py", "ref_gatne_v1")


def gcn_train_eval():
    """GCN/train_eval.py (the reference training loop: Adam, cross-entropy, one full-graph step per epoch)."""
    with folder("GCN"):
        return load_file("GCN/train_eval.py", "ref_gcn_train_eval")


def sage_data_utils():
    """GraphSAGE_Pytorch/data_utils.py (collate_fn: the sampler + the python-list feature gather)."""
    with folder("GraphSAGE_Pytorch"):
        importlib.import_module("sample_utils")
        return load_file("GraphSAGE_Pytorch/data_utils.py", "ref_sage_data_utils")


def gtn():
    """GTN/models package (GTN_Model, norm, GTLayer, GTConv)."""
    with folder("GTN"):
        m = importlib.import_module("models.GTN")
        return {"GTN": m, "GTLayer": importlib.import_module("models.GTLayer"),
                "GTConv": importlib.import_module("models.GTConv")}
