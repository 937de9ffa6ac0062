"""CPU: the oracle (oracle/mpnn_oracle.py) against the golden fixtures produced by the
unmodified reference (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import mpnn_oracle as O
from tests.conftest import GOLDEN, MODELS, load_gdb13, load_small, pretrained_like_state_dict

LOGIT_TOL = 1e-5      # fp32 re-association noise only (observed <= 1e-6)
GRAD_REL_TOL = 1e-5


@pytest.mark.parametrize("model", MODELS)
def test_oracle_matches_golden_logits_loss_grads(model):
    fx = load_small(model)
    loss, out, grads = O.train_step_grads(fx["sd"], fx["C"], fx["nodes"], fx["edges"], fx["target"])
    assert (out - fx["logits"]).abs().max().item() <= LOGIT_TOL
    assert torch.equal(out.argmax(1), fx["logits"].argmax(1))
    assert abs(float(loss) - fx["loss"]) <= 1e-6
    for k, g in fx["grads"].items():
        scale = max(g.abs().max().item(), 1e-12)
        assert (grads[k] - g).abs().max().item() / scale <= GRAD_REL_TOL, k


@pytest.mark.parametrize("model", MODELS)
def test_param_schema_matches_reference_state_dict(model):
    fx = load_small(model)
    shapes = O.param_shapes(fx["C"])
    assert [k for k, _ in shapes] == list(fx["sd"].keys())
    assert all(tuple(fx["sd"][k].shape) == tuple(s) for k, s in shapes)
    sd = O.init_state_dict(fx["C"], seed=1)
    assert list(sd.keys()) == list(fx["sd"].keys())


def test_oracle_pretrained_gdb13_rows():
    fx = load_gdb13()
    C = O.make_constants("GGNN")
    out = O.forward(pretrained_like_state_dict(), C, fx["nodes"], fx["edges"])
    assert (out.reshape(-1)[fx["logit_index"]] - fx["logit_sample"]).abs().max().item() <= 2e-5
    assert torch.equal(out.argmax(1), fx["argmax"])
    loss = O.kl_loss(out, fx["apds"])
    assert abs(float(loss) - fx["loss"]) <= 1e-5


def test_kl_loss_matches_definition():
    torch.manual_seed(0)
    out = torch.randn(7, 33)
    t = torch.rand(7, 33)
    t[0, :5] = 0
    th = t / t.sum(1, keepdim=True)
    want = (torch.xlogy(th, th) - th * torch.log_softmax(out, 1)).sum() / 7
    assert abs(float(O.kl_loss(out, t)) - float(want)) < 1e-6


def _live():
    return np.load(os.path.join(GOLDEN, "live_reference.npz"))


@pytest.mark.parametrize("model", MODELS)
def test_oracle_matches_live_reference(model):
    """molecules the small fixtures do not hold, through the reference as recorded by tests/golden/make_golden.py"""
    from graphinvent_b200 import synthetic as S
    fx = load_small(model)
    C = fx["C"]
    n, e = S.random_graphs(24, C.max_n_nodes, 4, 2, seed=77, min_atoms=0)
    nodes, edges = torch.from_numpy(n).float(), torch.from_numpy(e).float()
    with torch.no_grad():
        out = O.forward(fx["sd"], C, nodes, edges)
    assert (out - torch.from_numpy(_live()[f"logits/{model}"])).abs().max().item() <= LOGIT_TOL


@pytest.mark.parametrize("model", MODELS)
def test_oracle_training_curve_follows_the_reference(model):
    """50 steps of Workflow.train_epoch (Adam + OneCycleLR) with the oracle's functional forward against the curve
    of the unmodified reference (tests/golden/make_loss_curves.py); SURVEY.md 8c tolerance 1e-4"""
    import os

    import numpy as np
    from tests.conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, "loss_curves.npz"))
    fx = load_small(model)
    sd = {k: torch.nn.Parameter(v.clone()) for k, v in fx["sd"].items()}
    steps = int(z["steps"])
    opt = torch.optim.Adam(list(sd.values()), lr=float(z["lr"]))
    sch = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=float(z["max_lr"]), total_steps=steps)
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        loss = O.kl_loss(O.forward(sd, fx["C"], fx["nodes"], fx["edges"]), fx["target"])
        loss.backward()
        opt.step()
        sch.step()
        losses.append(loss.item())
    dev = np.abs(np.array(losses) - z[f"loss/{model}"])
    assert dev[0] <= 1e-6 and dev.max() <= 1e-4, (model, float(dev.max()))


def _multitype_batch(C):
    """two 3-atom molecules; the second carries a bond with two non-zero types (slot 0 of a generation batch
    accumulates such bonds, GraphGenerator.py:418-423)"""
    B, N, F, Ef = 2, C.max_n_nodes, C.n_node_features, C.n_edge_features
    nodes = torch.zeros(B, N, F)
    edges = torch.zeros(B, N, N, Ef)
    nodes[:, :3, 0] = 1
    edges[0, 0, 1, 0] = edges[0, 1, 0, 0] = 1
    edges[0, 1, 2, 1] = edges[0, 2, 1, 1] = 1
    edges[1, 0, 1, 0] = edges[1, 1, 0, 0] = 1
    edges[1, 0, 1, 2] = edges[1, 1, 0, 2] = 1
    return nodes, edges


def test_reference_aggregation_mpnn_rejects_multi_type_bonds():
    """error behaviour the drop-in mirrors: the reference's AggregationMPNN prologue sizes the neighbour slots by the
    summed bond VALUES (aggregation_mpnn.py:115-141), so a bond with two non-zero types makes its index assignment
    raise -- AttentionGGNN does not accept such input in the reference either.  The oracle follows the reference
    on both sides."""
    z = _live()
    assert str(z["multitype_error/AttGGNN"]).startswith("RuntimeError")
    C = O.make_constants("AttGGNN")
    nodes, edges = _multitype_batch(C)
    with pytest.raises(RuntimeError):
        O.forward(O.init_state_dict(C, seed=2), C, nodes, edges)
    for model in ("GGNN", "MNN"):                           # the summation family handles it (sum over the types)
        ref = torch.from_numpy(z[f"multitype_logits/{model}"])
        assert torch.isfinite(ref).all()
        Cs = O.make_constants(model)
        out = O.forward(O.init_state_dict(Cs, seed=2), Cs, nodes, edges)
        assert (out - ref).abs().max().item() <= LOGIT_TOL, model


def test_reference_edge_mpnn_rejects_multi_type_bonds():
    """the reference's EMN fails on such a bond too: `edge_degrees` sums the bond VALUES (edge_mpnn.py:123) while the
    incoming-edge lists come from `nonzero()` (:118-121), so the comparison at :156 raises a shape mismatch.  In the
    reference generator this state is reachable only in the never-reset dummy graph of slot 0 (INTEGRATION.md 2) -- the
    reason `tools/bench_generation.py` retries seeds for its CPU leg.  The oracle fails on it as well."""
    assert str(_live()["multitype_error/EMN"]).startswith("RuntimeError")
    C = O.make_constants("EMN")
    nodes, edges = _multitype_batch(C)
    with pytest.raises((RuntimeError, IndexError)):
        O.forward(O.init_state_dict(C, seed=2), C, nodes, edges)
