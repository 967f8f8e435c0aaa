"""Import the UNMODIFIED reference modules.  TEST INFRASTRUCTURE (oracle/__init__.py).

The reference (the original DeepRecommendation project) is not part of this repository: B200REC_REFERENCE_ROOT names a
checkout of it.  Only `make_golden.py` and the tests marked `reference` use this; those tests skip when it is not set.
"""
import importlib
import os
import sys

REFERENCE_ROOT = os.environ.get('B200REC_REFERENCE_ROOT', '')
_SRC = os.path.join(REFERENCE_ROOT, 'src')
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'pyg_shim')


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(_SRC, 'neural_collaborative_filtering'))


def _ensure_path():
    if not available():
        raise RuntimeError(f'reference not found: set B200REC_REFERENCE_ROOT to a checkout of the original project (now {REFERENCE_ROOT!r})')
    try:
        import torch_geometric  # noqa: F401  (a real install wins over the shim)
    except ImportError:
        if _SHIM not in sys.path:
            sys.path.insert(0, _SHIM)
    if _SRC not in sys.path:
        sys.path.insert(0, _SRC)


def load():
    """Returns a namespace with the reference classes/functions on the hot path."""
    _ensure_path()
    ns = type('reference', (), {})()
    ns.BasicNCF = importlib.import_module('neural_collaborative_filtering.models.basic_ncf').BasicNCF
    att = importlib.import_module('neural_collaborative_filtering.models.attention_ncf')
    ns.AttentionNCF = att.AttentionNCF
    gnn = importlib.import_module('neural_collaborative_filtering.models.gnn_ncf')
    ns.GraphNCF, ns.LightGCNConv, ns.LightGATConv = gnn.GraphNCF, gnn.LightGCNConv, gnn.LightGATConv
    ns.build_MLP_layers = importlib.import_module('neural_collaborative_filtering.util').build_MLP_layers
    ns.create_graph = importlib.import_module('content_providers.graph_providers').create_graph
    ns.DynamicProfilesProvider = importlib.import_module(
        'content_providers.dynamic_profiles_provider').DynamicProfilesProvider
    ns.datasets_fixed = importlib.import_module('neural_collaborative_filtering.datasets.fixed_datasets')
    ns.datasets_dynamic = importlib.import_module('neural_collaborative_filtering.datasets.dynamic_datasets')
    ns.datasets_gnn = importlib.import_module('neural_collaborative_filtering.datasets.gnn_datasets')
    ns.checkpoint_dir = os.path.join(REFERENCE_ROOT, 'models', 'runs')
    return ns
