"""CPU suite, part 4: the reference's CONSUMERS of the hot path run unchanged.

`models/gcn.py` and `experiment/training_loop.py` are imported from /root/reference without edits, on the
`torch_geometric` stand-in, and trained on a synthetic node-classification task over a graph in exactly the form the
drop-in `rewire` returns (int64 `[2, 2E]`, `from_networkx` column order).  Skipped where the reference checkout is
absent (the GPU box); the GPU side of config 2 is `tests/test_gpu_dropin.py::test_config2_rewire_then_gcn_on_gpu`.
"""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

REFERENCE = "/root/reference"


def _import_reference_consumers():
    from dcr import compat
    compat.ensure_torch_geometric()
    if REFERENCE not in sys.path:
        sys.path.append(REFERENCE)          # AFTER the package: rewiring/curvature/utils stay ours, the rest merges
    gcn = importlib.import_module("models.gcn")
    loop = importlib.import_module("experiment.training_loop")
    assert gcn.__file__.startswith(REFERENCE) and loop.__file__.startswith(REFERENCE)
    return gcn, loop


def _synthetic_task(n, edge_index, classes=3, feats=16, seed=0):
    from torch_geometric.data import Data, InMemoryDataset
    g = torch.Generator().manual_seed(seed)
    y = torch.randint(0, classes, (n,), generator=g)
    x = torch.randn(n, feats, generator=g) + 2.0 * torch.nn.functional.one_hot(y, classes).float() @ torch.randn(
        classes, feats, generator=g)
    perm = torch.randperm(n, generator=g)
    masks = {k: torch.zeros(n, dtype=torch.bool) for k in ("train_mask", "val_mask", "test_mask")}
    masks["train_mask"][perm[: n // 2]] = True
    masks["val_mask"][perm[n // 2: 3 * n // 4]] = True
    masks["test_mask"][perm[3 * n // 4:]] = True
    data = Data(x=x, edge_index=edge_index, y=y, **masks)
    return InMemoryDataset(data, num_classes=classes), data


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, "models")), reason="reference checkout absent")
def test_reference_gcn_and_training_loop_run_unchanged_on_rewired_graph():
    gcn, loop = _import_reference_consumers()
    from dcr.synth import named_graph
    from oracle.sdrf import sdrf_oracle
    ei, n = named_graph("texas")
    uni = np.random.RandomState(0).random_sample(10)
    rewired, _ = sdrf_oracle(ei, n, 10, True, 1.64, 22, uni)          # what rewire(...) returns, computed on the CPU
    assert rewired.shape[0] == 2 and rewired.dtype == np.int64
    dataset, data = _synthetic_task(n, torch.from_numpy(rewired))
    torch.manual_seed(0)
    model = gcn.GCN(dataset, hidden=[32], dropout=0.2)
    opt = torch.optim.Adam([{"params": model.non_reg_params, "weight_decay": 0},
                            {"params": model.reg_params, "weight_decay": 0.01}], lr=0.05)
    before = loop.evaluate(model, data, test=True)
    model = loop.training_loop(model, opt, data, epochs=40, patience=40)
    after = loop.evaluate(model, data, test=True)
    assert after["val_acc"] >= before["val_acc"]
    assert after["val_acc"] > 0.6 and after["test_acc"] > 0.5


def test_gcnconv_standin_matches_dense_formula():
    from dcr import compat
    compat.ensure_torch_geometric()
    from torch_geometric.nn import GCNConv
    torch.manual_seed(1)
    n = 12
    A = (torch.rand(n, n) < 0.3).float()
    A = ((A + A.t()) > 0).float()
    A.fill_diagonal_(0)
    ei = A.nonzero().t().contiguous()
    conv = GCNConv(5, 4)
    x = torch.randn(n, 5)
    Ah = A + torch.eye(n)
    dinv = Ah.sum(1).pow(-0.5)
    want = (dinv[:, None] * Ah * dinv[None, :]) @ (x @ conv.weight.t()) + conv.bias
    assert torch.allclose(conv(x, ei), want, atol=1e-5)
