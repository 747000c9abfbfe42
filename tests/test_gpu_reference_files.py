"""The reference's OWN model files, unmodified, running on the drop-in modules on the GPU.

Needs oracle/_ref/reference.zip (made by __graft_entry__.build() where a checkout of the reference is at hand --
oracle/refarchive.py) and is skipped without it: the reference's sources are not part of this repository.

  * install(fused_models=False): model/graph/{LightGCN,XSimGCL,SimGCL}.py are imported from the reference tree
    and trained for the three recorded batches of tests/golden/train_*.npz (same initial tables, same batches,
    same noise draws); the parameters must equal the ones the reference produced on its own stack (1e-4).
  * install() (default, fused models): the reference's DirectAU.py -- which imports LGCN_Encoder /
    Matrix_Factorization from model.graph.LightGCN / model.graph.MF (DirectAU.py:6-7) -- trains end to end.
"""
import importlib
import os
import random
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CFG = {
    "LightGCN": {"n_layer": 3},
    "SimGCL": {"n_layer": 2, "lambda": 0.5, "eps": 0.1},
    "XSimGCL": {"n_layer": 3, "l_star": 1, "lambda": 0.2, "eps": 0.2, "tau": 0.2},
}
TOP = ("base", "util", "data", "model")


@pytest.fixture(scope="module")
def ref_root(tmp_path_factory, built_lib):
    import torch
    assert torch.cuda.is_available()
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refarchive
    if not refarchive.available():
        pytest.skip("oracle/_ref/reference.zip is absent (build() makes it where a checkout of the reference is at hand)")
    return refarchive.unpack(str(tmp_path_factory.mktemp("reference")))


@pytest.fixture()
def reference_imports(ref_root):
    """Import state of a reference checkout: its root first on sys.path, no stale base/util/data/model modules."""
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in TOP}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, ref_root)
    yield ref_root
    sys.path.remove(ref_root)
    for k in [k for k in sys.modules if k.split(".")[0] in TOP]:
        del sys.modules[k]
    sys.modules.update(saved)


@pytest.mark.parametrize("name", ["LightGCN", "XSimGCL", "SimGCL"])
def test_reference_model_file_trains_on_the_dropins(reference_imports, golden, tiny_conf, tiny_triples, in_tmp_cwd, monkeypatch, name):
    import torch
    import selfrec_b200
    selfrec_b200.install(fused_models=False)
    mod = importlib.import_module(f"model.graph.{name}")
    assert os.path.realpath(mod.__file__).startswith(os.path.realpath(reference_imports)), "the reference's own file must be the one imported"
    assert sys.modules["util.loss_torch"].__name__.startswith("selfrec_b200"), "the losses must be the drop-ins"
    fx = golden(f"train_{name}.npz")
    train, test = tiny_triples
    torch.manual_seed(0)
    m = getattr(mod, name)(tiny_conf(name, CFG[name]), [list(t) for t in train], [list(t) for t in test])
    with torch.no_grad():
        m.model.embedding_dict["user_emb"].copy_(torch.from_numpy(fx["init_user"]))
        m.model.embedding_dict["item_emb"].copy_(torch.from_numpy(fx["init_item"]))
    n_steps = int(fx["n_steps"])

    def recorded_batches(data, batch_size, n_negs=1):
        for k in range(n_steps):
            yield tuple(fx[f"b{k}_{t}"].tolist() for t in ("u", "i", "j"))

    monkeypatch.setattr(mod, "next_batch_pairwise", recorded_batches)
    if "noise" in fx.files:  # the reference draws torch.rand_like(...) per perturbed layer: hand it the recorded draws
        draws = iter(fx["noise"])
        monkeypatch.setattr(torch, "rand_like", lambda t, *a, **k: torch.from_numpy(next(draws)).to(t.device))
    m.maxEpoch = 1
    m.train()
    got = torch.cat([m.model.embedding_dict["user_emb"], m.model.embedding_dict["item_emb"]]).detach().cpu().numpy()
    np.testing.assert_allclose(got, fx[f"params_after_{n_steps - 1}"], rtol=1e-4, atol=1e-6)
    assert m.bestPerformance, "fast_evaluation ran on the drop-in test() path"
    # the adjacency handle the reference's encoder holds is the CUDA CSR, not a torch COO tensor
    from selfrec_b200.ops import SparseAdj
    assert isinstance(m.model.sparse_norm_adj, SparseAdj)


def test_reference_directau_runs_end_to_end_with_the_default_install(reference_imports, tiny_conf, tiny_triples, in_tmp_cwd):
    """SURVEY 8(f) row 4: a LightGCN-backbone model outside the five fused ones, unmodified, on the default install
    (its `from model.graph.LightGCN import LGCN_Encoder` resolves to the drop-in encoder)."""
    import torch
    import selfrec_b200
    selfrec_b200.install()
    mod = importlib.import_module("model.graph.DirectAU")
    assert os.path.realpath(mod.__file__).startswith(os.path.realpath(reference_imports))
    assert mod.LGCN_Encoder.__module__.startswith("selfrec_b200") and mod.Matrix_Factorization.__module__.startswith("selfrec_b200")
    train, test = tiny_triples
    random.seed(3)
    torch.manual_seed(3)
    m = mod.DirectAU(tiny_conf("DirectAU", {"gamma": 2, "n_layers": 2}, **{"max.epoch": 3}), [list(t) for t in train], [list(t) for t in test])
    before = torch.cat([p.detach().clone().flatten() for p in m.model.parameters()])
    m.train()
    after = torch.cat([p.detach().flatten() for p in m.model.parameters()])
    assert torch.isfinite(after).all() and (after - before.to(after.device)).abs().max() > 1e-4
    assert len(m.bestPerformance) == 2 and set(m.bestPerformance[1]) >= {"Hit Ratio", "Precision", "Recall", "NDCG"}
    rec = m.test()
    assert len(rec) > 0 and all(len(v) == m.max_N for v in rec.values())
