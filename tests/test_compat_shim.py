"""The torch_geometric import shim exposes, backed by this package, the names SpotV2Net's own modules import."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def shim_on_path():
    compat = os.path.join(ROOT, "compat")
    saved = {k: v for k, v in sys.modules.items() if k == "torch_geometric" or k.startswith("torch_geometric.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, compat)
    yield compat
    sys.path.remove(compat)
    for k in [k for k in sys.modules if k == "torch_geometric" or k.startswith("torch_geometric.")]:
        del sys.modules[k]
    sys.modules.update(saved)


def test_shim_exposes_the_names_the_reference_imports(shim_on_path):
    import spotv2net_b200 as sv
    from torch_geometric.nn import GATConv, GATv2Conv
    from torch_geometric.loader import DataLoader
    from torch_geometric.data import Data
    assert GATConv is sv.GATConv and issubclass(DataLoader, sv.WindowLoader)
    with pytest.raises(NotImplementedError):
        GATv2Conv(4, 4)
    d = Data(x=torch.zeros(2, 3), edge_index=torch.zeros(2, 2, dtype=torch.long))
    assert d.x.shape == (2, 3)
    with pytest.raises(TypeError):
        DataLoader([1, 2, 3], batch_size=2)
