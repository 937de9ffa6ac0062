"""GPU: the drop-in modules (CUDA path through the C-ABI) against the oracle and the golden
fixtures of the unmodified reference.  Tolerances (north_star / SURVEY.md §8c):
   logits  max-abs <= 1e-4 vs CPU fp32, APD argmax identical,
   grads   per-tensor max|d| / max|g| <= 1e-4,
   loss    <= 1e-5."""
import copy
from collections import OrderedDict

import numpy as np
import pytest
import torch

from tests.conftest import MODELS, load_gdb13, load_small, pretrained_like_state_dict

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-4
GRAD_REL_TOL = 1e-4


def Fn_lib():
    from graphinvent_b200._lib import lib
    return lib


def _build(C, sd=None):
    from graphinvent_b200.gnn import mpnn
    net = mpnn.create(C)
    if sd is not None:
        net.load_state_dict(sd)
    return net.cuda()


def _step(net, nodes, edges, target):
    from graphinvent_b200 import functional as Fn
    net.zero_grad()
    out = net(nodes.cuda(), edges.cuda())
    loss = Fn.kl_loss(out, target.cuda())
    loss.backward()
    grads = OrderedDict((k, p.grad.detach().cpu()) for k, p in net.named_parameters())
    return out.detach().cpu(), float(loss), grads


KINK_L2_TOL = 2e-2    # batches that sit on SELU kinks: see _well_conditioned() and DESIGN.md


def _assert_grads(got, want, tol=GRAD_REL_TOL, l2=False):
    """per-tensor error relative to that tensor's gradient scale; tensors whose true gradient vanishes
    (e.g. the gather attention net on molecules without bonds: all energies tie, d softmax == 0) hold pure
    rounding noise in BOTH implementations, so the scale is floored at 1e-4 of the global gradient scale"""
    gmax = max(g.abs().max().item() for g in want.values())
    gnorm = max(g.norm().item() for g in want.values())
    worst = ("", 0.0)
    for k, g in want.items():
        if l2:
            rel = (got[k] - g).norm().item() / max(g.norm().item(), 1e-4 * gnorm, 1e-12)
        else:
            rel = (got[k] - g).abs().max().item() / max(g.abs().max().item(), 1e-4 * gmax, 1e-12)
        if rel > worst[1]:
            worst = (k, rel)
    assert worst[1] <= tol, f"worst gradient {worst[0]}: rel err {worst[1]:.3e} (tol {tol:g})"


def _margins(C, sd, nodes, edges):
    """per-molecule distance of the closest SELU input / masked gather energy to a point where the path is
    not differentiable / not continuous (oracle MARGINS probe); NaN where the reference cannot run the
    molecule on its own (AttentionGGNN / EMN on a bond-less batch)."""
    from oracle import mpnn_oracle as O
    out = []
    try:
        with torch.no_grad():
            for b in range(nodes.shape[0]):
                O.MARGINS = []
                try:
                    O.forward(sd, C, nodes[b:b + 1], edges[b:b + 1])
                    out.append(min(O.MARGINS))
                except RuntimeError:
                    out.append(float("nan"))
    finally:
        O.MARGINS = None
    return torch.tensor(out, dtype=torch.float64)


def _well_conditioned(C, sd, nodes, edges, margin=8e-6, n_bonded=40, n_bondless=8):
    """Indices of the best-conditioned molecules (stratified: with and without bonds).  fp32 rounding noise
    between two correct implementations is ~1e-6 on the SELU inputs, so on molecules whose margin is >= 8e-6
    a correct CUDA path must meet the strict tolerance; on arbitrary batches the reference itself moves by up
    to 7e-3 between fp32 and fp64 (measured, DESIGN.md "numerical conditioning")."""
    m = _margins(C, sd, nodes, edges)
    bonded = edges.sum((1, 2, 3)) > 0
    keep = []
    for mask, cap in ((bonded, n_bonded), (~bonded, n_bondless)):
        idx = torch.nonzero(mask & (m >= margin)).flatten()
        idx = idx[torch.argsort(m[idx], descending=True)][:cap]
        keep += sorted(idx.tolist())
    return torch.tensor(keep, dtype=torch.long)


@pytest.mark.parametrize("model", MODELS)
def test_golden_small_forward_backward(model):
    """fixture = unmodified reference on CPU (tests/golden/make_golden.py); includes the generator's corner
    graphs: dummy self-loop graph, empty graph, isolated atom, degree-5 atom."""
    fx = load_small(model)
    net = _build(fx["C"], fx["sd"])
    assert list(net.state_dict().keys()) == list(fx["sd"].keys())
    out, loss, grads = _step(net, fx["nodes"], fx["edges"], fx["target"])
    assert torch.isfinite(out).all()
    assert (out - fx["logits"]).abs().max().item() <= LOGIT_TOL
    assert torch.equal(out.argmax(1), fx["logits"].argmax(1))
    assert abs(loss - fx["loss"]) <= 1e-5
    _assert_grads(grads, fx["grads"])


@pytest.mark.parametrize("model", MODELS)
def test_default_dims_vs_oracle(model):
    """reference default hyper-parameters (defaults.py:145-433), gdb13 chemistry, real-data-like sizes"""
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    C = O.make_constants(model)
    sd = O.init_state_dict(C, seed=11)
    n, e = S.random_graphs(96, 13, 5, 3, seed=12, min_atoms=0)
    n2, e2 = S.corner_case_graphs(13, 8)
    nodes = torch.from_numpy(np.concatenate([n2, n])).float()
    edges = torch.from_numpy(np.concatenate([e2, e])).float()
    target = torch.from_numpy(S.random_targets(nodes.shape[0], 625, seed=3))
    loss_ref, out_ref, g_ref = O.train_step_grads(sd, C, nodes, edges, target)
    net = _build(C, sd)
    out, loss, grads = _step(net, nodes, edges, target)
    assert (out - out_ref).abs().max().item() <= LOGIT_TOL
    assert torch.equal(out.argmax(1), out_ref.argmax(1))
    assert abs(loss - float(loss_ref)) <= 1e-5
    # an arbitrary batch sits on SELU kinks (8e6 activations, margins down to 1e-7): gradients are only
    # comparable in norm here; the strict gradient check is the well-conditioned test below
    _assert_grads(grads, g_ref, tol=KINK_L2_TOL, l2=True)


@pytest.mark.parametrize("model", MODELS)
def test_default_dims_strict_gradients_on_well_conditioned_molecules(model):
    """default hyper-parameters, molecules selected (by the oracle's conditioning probe) to be away from
    the non-differentiable points of the path: logits AND every parameter gradient within 1e-4."""
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    C = O.make_constants(model)
    # parameter seeds chosen so that the constant activation chains every molecule shares (all-zero padding
    # slots, zero initial edge memories) are themselves >= 8e-6 away from a SELU kink
    sd = O.init_state_dict(C, seed={"AttGGNN": 16, "EMN": 16}.get(model, 11))
    n, e = S.random_graphs(1500, 13, 5, 3, seed=21, min_atoms=0)
    n2, e2 = S.corner_case_graphs(13, 8)
    nodes = torch.from_numpy(np.concatenate([n2, n])).float()
    edges = torch.from_numpy(np.concatenate([e2, e])).float()
    keep = _well_conditioned(C, sd, nodes, edges)
    n_bonded = int((edges[keep].sum((1, 2, 3)) > 0).sum())
    assert n_bonded >= 12, f"only {n_bonded} well-conditioned molecules with bonds"
    nodes, edges = nodes[keep], edges[keep]
    target = torch.from_numpy(S.random_targets(nodes.shape[0], 625, seed=5))
    loss_ref, out_ref, g_ref = O.train_step_grads(sd, C, nodes, edges, target)
    out, loss, grads = _step(_build(C, sd), nodes, edges, target)
    assert (out - out_ref).abs().max().item() <= LOGIT_TOL
    assert torch.equal(out.argmax(1), out_ref.argmax(1))
    assert abs(loss - float(loss_ref)) <= 1e-5
    _assert_grads(grads, g_ref)


def test_pretrained_checkpoint_on_real_gdb13_rows():
    """weights with the shipped checkpoint's layout and per-tensor statistics (conftest.pretrained_like_state_dict)
    x the first 256 real rows of gdb13_1K/train.h5; golden loss / argmax / sampled logits / gradient statistics from
    the unmodified reference."""
    from oracle import mpnn_oracle as O
    fx = load_gdb13()
    net = _build(O.make_constants("GGNN"), pretrained_like_state_dict())     # reference layout loads unchanged
    out, loss, grads = _step(net, fx["nodes"], fx["edges"], fx["apds"])
    idx = fx["logit_index"]
    err = (out.reshape(-1)[idx] - fx["logit_sample"]).abs()
    bonded = (fx["edges"].sum((1, 2, 3)) > 0)
    on_bonded = bonded[idx // out.shape[1]]
    print(f"pretrained-like/gdb13: max sampled logit err bonded {err[on_bonded].max().item():.3e}, bond-less "
          f"{err[~on_bonded].max().item() if (~on_bonded).any() else 0:.3e}, tensor cores {Fn_lib().gib_get_tensor_cores()}")
    assert err[on_bonded].max().item() <= LOGIT_TOL, f"bonded molecules: {err[on_bonded].max().item():.3e}"
    # molecules without a bonded atom: the reference rounds `energies - 1e6` to multiples of 1/16 in fp32, so a
    # 1e-6 difference upstream can land in another bucket (reference fp32 vs fp64: 3.3e-3 on such rows,
    # BASELINE.md §2); well-conditioned bond-less molecules are held to 1e-4 in the strict default-dims test.
    if (~on_bonded).any():
        assert err[~on_bonded].max().item() <= 2e-2, f"bond-less molecules: {err[~on_bonded].max().item():.3e}"
    assert torch.equal(out.argmax(1)[bonded], fx["argmax"][bonded])
    assert abs(loss - fx["loss"]) <= 1e-4
    g = fx["g"]
    # gradient statistics / a few full gradients recorded from the unmodified reference.  256 arbitrary
    # real rows sit on SELU kinks, so these are norm-level checks; the strict comparison follows.
    names = [str(s) for s in g["grad_names"]]
    for k, amax in zip(names, g["grad_absmax"]):
        assert abs(grads[k].abs().max().item() - float(amax)) <= KINK_L2_TOL * max(float(amax), 1e-9), k
    for k in g.files:
        if k.startswith("grad/"):
            want = torch.from_numpy(g[k])
            assert (grads[k[5:]] - want).norm().item() <= KINK_L2_TOL * max(want.norm().item(), 1e-12), k
    # (no strict subset here: with the shipped trained weights the all-zero padding slots themselves sit
    #  6e-7 from a SELU kink, so every real row is ill-conditioned; the strict gradient comparison is
    #  test_default_dims_strict_gradients_on_well_conditioned_molecules)


def test_bond_values_other_than_one_and_multi_type_bonds():
    """GGNN / MNN follow the reference arithmetic for arbitrary non-negative bond values
    (mpnn.py:284-294: value * MLP_t(value * h)); AttentionGGNN refuses multi-type bonds loudly."""
    from oracle import mpnn_oracle as O
    for model in ("GGNN", "MNN"):
        fx = load_small(model)
        edges = fx["edges"].clone()
        edges[6, 0, 1, :] = torch.tensor([0.5, 0.0, 2.0]); edges[6, 1, 0, :] = torch.tensor([0.5, 0.0, 2.0])
        edges[7] *= 1.5
        out_ref = O.forward(fx["sd"], fx["C"], fx["nodes"], edges)
        net = _build(fx["C"], fx["sd"])
        with torch.no_grad():
            out = net(fx["nodes"].cuda(), edges.cuda()).cpu()
        assert (out - out_ref).abs().max().item() <= LOGIT_TOL, model
    fx = load_small("AttGGNN")
    edges = fx["edges"].clone()
    edges[6, 0, 1, :] = 1.0
    with pytest.raises(RuntimeError, match="one bond type"):
        _build(fx["C"], fx["sd"])(fx["nodes"].cuda(), edges.cuda())


def test_module_protocol_eval_nograd_deepcopy_statedict_reentrancy():
    """what Workflow / GraphGenerator / the RL loop do with the module (SURVEY.md §8b)."""
    from graphinvent_b200 import functional as Fn
    fx = load_small("GGNN")
    net = _build(fx["C"], fx["sd"])
    nodes, edges, tgt = fx["nodes"].cuda(), fx["edges"].cuda(), fx["target"].cuda()
    net.eval()
    with torch.no_grad():
        o1 = net(nodes, edges)
    net.train()
    o2 = net(nodes, edges)
    assert torch.equal(o1, o2)                                   # p = 0 dropout: identical; bit-stable kernels
    twin = copy.deepcopy(net)                                    # Workflow.py:187-188
    assert torch.equal(twin(nodes, edges), o2)
    sd = net.state_dict()
    assert all(torch.equal(sd[k].cpu(), fx["sd"][k]) for k in fx["sd"])
    # RL-style: several forwards, one backward (Workflow.py:582-598)
    net.zero_grad()
    l1 = Fn.kl_loss(net(nodes[:16], edges[:16]), tgt[:16])
    l2 = Fn.kl_loss(net(nodes[16:], edges[16:]), tgt[16:])
    (l1 * 16 + l2 * 16).div(32).backward()
    g_two = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    Fn.kl_loss(net(nodes, edges), tgt).backward()
    for a, b in zip(g_two, net.parameters()):
        assert (a - b.grad).abs().max().item() <= 1e-5 * max(1.0, b.grad.abs().max().item())
    # optimizer step changes the weights -> packed copy must refresh
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    opt.step()
    o3 = net(nodes, edges)
    assert not torch.equal(o3, o2)
    # varying batch size (last batch, generation)
    assert net(nodes[:1], edges[:1]).shape == (1, o2.shape[1])
    assert (net(nodes[:3], edges[:3]) - o3[:3]).abs().max().item() <= 2e-5


def test_batch_without_any_bond_does_not_break_the_kernels():
    """zero bond entries (P = 0): every per-entry kernel / GEMM gets an empty row range; forward and backward must
    still run and give finite values (the reference generator avoids this case with its dummy graph)"""
    from graphinvent_b200 import functional as Fn
    for model in MODELS:
        fx = load_small(model)
        net = _build(fx["C"], fx["sd"])
        nodes = fx["nodes"][1:3].cuda()                    # the empty graph and the isolated atom
        edges = torch.zeros_like(fx["edges"][1:3]).cuda()
        out = net(nodes, edges)
        Fn.kl_loss(out, fx["target"][1:3].cuda()).backward()
        assert torch.isfinite(out).all(), model
        assert all(torch.isfinite(p.grad).all() for p in net.parameters()), model
        if model in ("GGNN", "MNN"):                       # the reference can run these two on a bond-less batch
            from oracle import mpnn_oracle as O
            ref = O.forward(fx["sd"], fx["C"], nodes.cpu(), edges.cpu())
            assert (out.detach().cpu() - ref).abs().max().item() <= 2e-2   # mask-quantisation regime (DESIGN.md 4)


def test_int8_inputs_are_widened_on_the_device():
    """§8f rank 3: int8 batches (the reference's on-disk dtype) go to the device as 1 byte per element"""
    fx = load_small("GGNN")
    net = _build(fx["C"], fx["sd"])
    with torch.no_grad():
        a = net(fx["nodes"].cuda(), fx["edges"].cuda())
        b = net(fx["nodes"].to(torch.int8).cuda(), fx["edges"].to(torch.int8).cuda())
    assert torch.equal(a, b)


def test_cpu_tensors_fail_loudly():
    fx = load_small("GGNN")
    from graphinvent_b200.gnn import mpnn
    net = mpnn.create(fx["C"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(fx["nodes"], fx["edges"])


def test_attggnn_c3_shape_properties():
    """BASELINE configs[2] at full size (AttentionGGNN hidden=256, 6 passes, batch 2048 of 40-atom molecules):
    oracle-checked logits on a slice, sub-batch consistency, finite gradients for every parameter."""
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    C = O.make_constants("AttGGNN", hidden_node_features=256, message_size=256, message_passes=6, max_n_nodes=40,
                         n_node_features=12, len_f_add_per_node=81)
    apd = 40 * (81 + 3) + 1
    sd = O.init_state_dict(C, seed=3)
    n, e = S.random_graphs(2048, 40, 9, 3, seed=1003)
    nodes, edges = torch.from_numpy(n).float().cuda(), torch.from_numpy(e).float().cuda()
    target = torch.from_numpy(S.random_targets(2048, apd, seed=4)).cuda()
    net = _build(C, sd)
    out = net(nodes, edges)
    Fn.kl_loss(out, target).backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in net.parameters())
    with torch.no_grad():
        part = net(nodes[64:128], edges[64:128])
    assert (out[64:128] - part).abs().max().item() <= 5e-5      # sub-batch may route GEMMs to other kernels
    k = 24
    ref = O.forward(sd, C, nodes[:k].cpu(), edges[:k].cpu())
    assert (out[:k].detach().cpu() - ref).abs().max().item() <= LOGIT_TOL
    assert torch.equal(out[:k].detach().cpu().argmax(1), ref.argmax(1))


@pytest.mark.parametrize("cfg", ["C2", "C4"])
def test_full_size_properties(cfg):
    """BASELINE.json sizes, where the CPU oracle is too slow to be the checker: size-independent
    properties of the path -- (1) molecules are independent, so any sub-batch reproduces its rows
    bit-exactly; (2) permuting the batch permutes the logits; (3) gradients are additive over a
    partition of the batch; (4) one oracle-checked slice."""
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    if cfg == "C2":
        C = O.make_constants("GGNN", hidden_node_features=128, message_size=128, message_passes=4)
        B, N, na, nc = 1024, 13, 5, 3
    else:
        C = O.make_constants("GGNN", max_n_nodes=38, n_node_features=12, len_f_add_per_node=81)
        B, N, na, nc = 4096, 38, 9, 3
    apd = N * (C.len_f_add_per_node + C.len_f_conn_per_node) + 1
    sd = O.init_state_dict(C, seed=0)
    n, e = S.random_graphs(B, N, na, nc, seed=1002)
    nodes, edges = torch.from_numpy(n).float().cuda(), torch.from_numpy(e).float().cuda()
    target = torch.from_numpy(S.random_targets(B, apd, seed=2)).cuda()
    net = _build(C, sd)
    with torch.no_grad():
        full = net(nodes, edges)
        half = net(nodes[B // 2:], edges[B // 2:])
        perm = torch.randperm(B, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
        permuted = net(nodes[perm], edges[perm])
    assert torch.isfinite(full).all()
    # molecules are independent: a sub-batch reproduces its rows (bit-exactly on the SIMT path; the tcgen05 path may
    # route a GEMM to a different kernel when the row count changes, so allow fp32 rounding noise there)
    sub_err = (full[B // 2:] - half).abs().max().item()
    assert sub_err <= 2e-5, f"sub-batch vs full batch: {sub_err:.3e}"
    assert (permuted - full[perm]).abs().max().item() <= 1e-5   # type-grouped rows move between GEMM tiles
    assert torch.equal(permuted.argmax(1), full[perm].argmax(1))
    net.zero_grad()
    (Fn.kl_loss(net(nodes, edges), target)).backward()
    g_full = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    for sl in (slice(0, B // 2), slice(B // 2, B)):
        (Fn.kl_loss(net(nodes[sl], edges[sl]), target[sl]) * 0.5).backward()
    for a, p in zip(g_full, net.parameters()):
        # same function, different kernel routing / rounding for the half batches (and SELU-kink flips): norm-level
        assert (a - p.grad).norm().item() <= 2e-3 * max(a.norm().item(), 1e-6)
    k = 48
    out_ref = O.forward(sd, C, nodes[:k].cpu(), edges[:k].cpu())
    assert (full[:k].cpu() - out_ref).abs().max().item() <= LOGIT_TOL
    assert torch.equal(full[:k].cpu().argmax(1), out_ref.argmax(1))


# ------------------------------------------------------------------------------------------
# fp64-anchored parity on ARBITRARY batches (no oracle-selected inputs).  The yardstick is the reference's own fp32
# rounding -- the distance between the fp32 and the fp64 evaluation of the same expression -- plus the one thing
# rounding noise can legitimately change by more than noise: the side of 0 a SELU input falls on (SELU' jumps from
# 1.758 to 1.051 there).  That effect is COMPUTED, not assumed: the fp64 oracle is differentiated twice with the
# derivative of every SELU whose input lies within tau of 0 forced to its left / right limit (oracle KINK probe);
# ||g_L - g_R|| is the total gradient change the units inside the band can cause.  tau = a few times the forward
# rounding noise of the path (tensor cores: 3xTF32 products accumulate with truncation, measured logit deviation
# ~1e-5; fp32 SIMT GEMMs: ~5e-6).
#   gradients, per tensor:  ||g_cuda - g_fp64|| <= 2 ||g_ref32 - g_fp64|| + ||g_L(tau) - g_R(tau)|| + eps ||g_fp64||
#                           eps = 1e-6 with fp32 SIMT GEMMs; 3e-5 with tensor cores: the arithmetic of the 3xTF32 GEMMs
#                           themselves (dropped lo*lo term, truncating TMEM accumulation; measured against fp64 on random
#                           operands: 1e-6 .. 1e-5 of the largest entry, tools/gemm_check.py)
#   logits, per molecule:   max|o_cuda - o_fp64| <= 3 max|o_ref32 - o_fp64| + 1e-4
#   APD argmax:             identical to the fp32 reference wherever the reference's own top-2 gap exceeds its own
#                           fp32-vs-fp64 movement on that molecule (bond-less molecules included)
#   loss:                   |loss - loss_fp64| <= 3 |loss_ref32 - loss_fp64| + 1e-5 max(1, |loss|)
# ------------------------------------------------------------------------------------------
FP64_C = 3.0
KINK_TAU = {1: 3e-5, 0: 3e-6}      # tensor cores on / off
GEMM_EPS = {1: 3e-5, 0: 1e-6}


def _fp64_anchored(C, sd, nodes, edges, target, tag, tensor_cores=1):
    from oracle import mpnn_oracle as O
    lib = Fn_lib()
    l32, o32, g32 = O.train_step_grads(sd, C, nodes, edges, target)
    l64, o64, g64 = O.train_step_grads(sd, C, nodes, edges, target, dtype=torch.float64)
    tau = KINK_TAU[tensor_cores]
    try:
        O.KINK = (tau, "L")
        _, _, gL = O.train_step_grads(sd, C, nodes, edges, target, dtype=torch.float64)
        O.KINK = (tau, "R")
        _, _, gR = O.train_step_grads(sd, C, nodes, edges, target, dtype=torch.float64)
    finally:
        O.KINK = None
    lib.gib_set_tensor_cores(tensor_cores)
    try:
        out, loss, grads = _step(_build(C, sd), nodes, edges, target)
    finally:
        lib.gib_set_tensor_cores(1)
    # logits
    e_ref = (o32.double() - o64).abs().max(1).values
    e_cuda = (out.double() - o64).abs().max(1).values
    worst_row = ((e_cuda - FP64_C * e_ref - LOGIT_TOL).max().item())
    # argmax wherever the reference itself is decided
    top2 = o32.topk(2, dim=1).values
    decided = (top2[:, 0] - top2[:, 1]).double() > 2 * e_ref + 2 * LOGIT_TOL
    same = out.argmax(1) == o32.argmax(1)
    # gradients
    gscale = max(g.norm().item() for g in g64.values())
    worst = ("", 0.0, 0.0, 0.0, 0.0)
    tot = [0.0, 0.0, 0.0, 0.0]
    for k, g in g64.items():
        d_cuda = (grads[k].double() - g).norm().item()
        d_ref = (g32[k].double() - g).norm().item()
        d_kink = (gL[k] - gR[k]).norm().item()
        bound = 2.0 * d_ref + d_kink + GEMM_EPS[tensor_cores] * g.norm().item() + 1e-7 * gscale
        for i, v in enumerate((d_cuda, d_ref, d_kink, g.norm().item())):
            tot[i] += v * v
        if d_cuda / bound > worst[1]:
            worst = (k, d_cuda / bound, d_cuda, d_ref, d_kink)
    tot = [t ** 0.5 for t in tot]
    bondless = edges.sum((1, 2, 3)) == 0
    print(f"fp64-anchored [{tag}, tensor cores {tensor_cores}]: logits cuda-vs-fp64 {e_cuda.max().item():.2e} (ref32-vs-fp64 "
          f"{e_ref.max().item():.2e}), decided rows {int(decided.sum())}/{len(decided)} (bond-less "
          f"{int((decided & bondless).sum())}/{int(bondless.sum())}); gradients, global L2: |g| {tot[3]:.3e}, cuda-fp64 {tot[0]:.2e}, "
          f"ref32-fp64 {tot[1]:.2e}, kink band (tau {tau:g}) {tot[2]:.2e}; worst tensor {worst[0]}: {worst[1]:.2f} of its bound "
          f"(cuda {worst[2]:.2e}, ref32 {worst[3]:.2e}, kink {worst[4]:.2e}); loss {loss:.7f} vs fp64 {float(l64):.7f} / fp32 {float(l32):.7f}")
    assert worst_row <= 0, f"logits: a molecule moves {worst_row + LOGIT_TOL:.3e} beyond {FP64_C} x the reference's own fp32 error"
    assert bool(same[decided].all()), f"argmax differs on {int((~same & decided).sum())} molecules the reference decides"
    assert abs(loss - float(l64)) <= FP64_C * abs(float(l32) - float(l64)) + 1e-5 * max(1.0, abs(float(l64)))
    assert worst[1] <= 1.0, (f"gradient {worst[0]}: |cuda - fp64| = {worst[2]:.3e} exceeds 2 x |ref32 - fp64| = {worst[3]:.3e} "
                             f"+ kink band {worst[4]:.3e} (+ floor)")
    assert tot[0] <= 2.0 * tot[1] + tot[2] + GEMM_EPS[tensor_cores] * tot[3]


@pytest.mark.parametrize("tensor_cores", [1, 0])
@pytest.mark.parametrize("model", MODELS)
def test_fp64_anchored_default_dims_arbitrary_batch(model, tensor_cores):
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    C = O.make_constants(model)
    sd = O.init_state_dict(C, seed=11)
    n, e = S.random_graphs(96, 13, 5, 3, seed=12, min_atoms=0)
    n2, e2 = S.corner_case_graphs(13, 8)
    if model in ("AttGGNN", "EMN"):
        # the reference's AggregationMPNN / EdgeMPNN prologues need at least one bond in the batch; they have one here
        pass
    nodes = torch.from_numpy(np.concatenate([n2, n])).float()
    edges = torch.from_numpy(np.concatenate([e2, e])).float()
    target = torch.from_numpy(S.random_targets(nodes.shape[0], 625, seed=3))
    _fp64_anchored(C, sd, nodes, edges, target, f"{model} default dims, 101 molecules incl. corner graphs", tensor_cores)


def test_fp64_anchored_c2_slice():
    """BASELINE configs[1] model (GGNN hidden = message = 128, 4 passes) on 96 synthetic 13-atom molecules"""
    from graphinvent_b200 import synthetic as S
    from oracle import mpnn_oracle as O
    C = O.make_constants("GGNN", hidden_node_features=128, message_size=128, message_passes=4)
    sd = O.init_state_dict(C, seed=0)
    n, e = S.random_graphs(96, 13, 5, 3, seed=1002)
    nodes, edges = torch.from_numpy(n).float(), torch.from_numpy(e).float()
    target = torch.from_numpy(S.random_targets(96, 625, seed=1002))
    _fp64_anchored(C, sd, nodes, edges, target, "C2 model, 96 molecules")


def test_fp64_anchored_pretrained_on_all_real_gdb13_rows():
    """weights with the shipped checkpoint's per-tensor statistics x all 256 recorded real rows of gdb13_1K/train.h5
    (bonded and bond-less alike)"""
    from oracle import mpnn_oracle as O
    fx = load_gdb13()
    _fp64_anchored(O.make_constants("GGNN"), pretrained_like_state_dict(), fx["nodes"], fx["edges"], fx["apds"],
                   "pretrained-like weights x 256 real gdb13 rows")


def test_multi_type_bonds_follow_the_reference():
    """GGNN sums the per-type messages of a multi-type bond like the reference; AttentionGGNN raises, as the
    reference's AggregationMPNN does on such input (tests/test_oracle.py pins that against the live reference)"""
    from oracle import mpnn_oracle as O
    from tests.test_oracle import _multitype_batch
    C = O.make_constants("GGNN")
    sd = O.init_state_dict(C, seed=2)
    nodes, edges = _multitype_batch(C)
    ref = O.forward(sd, C, nodes, edges)
    with torch.no_grad():
        out = _build(C, sd)(nodes.cuda(), edges.cuda()).cpu()
    assert (out - ref).abs().max().item() <= LOGIT_TOL
    Ca = O.make_constants("AttGGNN")
    with pytest.raises(RuntimeError, match="one bond type per bond"):
        _build(Ca, O.init_state_dict(Ca, seed=2))(nodes.cuda(), edges.cuda())
