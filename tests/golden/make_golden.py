"""
Generates the golden fixtures in this directory by running the UNMODIFIED reference
(`graphinvent/gnn` of a GraphINVENT checkout, imported per SURVEY.md Appendix C) on CPU fp32:

    GRAPHINVENT_REFERENCE=<GraphINVENT checkout> python tests/golden/make_golden.py [part ...]

parts: small, gdb13, live (default: all).  Outputs
  small_<MODEL>.npz   tiny-dims config per model: constants (json), reference-initialised
                      state_dict, int8 inputs (random molecules + the generator's corner
                      graphs), targets, reference logits / loss / parameter gradients.
  gdb13_rows.npz      first 256 real rows of data/pre-training/gdb13_1K/train.h5 (int8).
  gdb13_train_excerpt.h5
                      that file cut to its 2048-byte header and its first 16 rows of each
                      dataset (same layout; for the raw HDF5 reader).
  checkpoint_stats.npz
                      name, shape, mean and standard deviation of every tensor of the shipped
                      GGNN checkpoint (data/fine-tuning/gdb13_1K-debug/pretrained_model.pth,
                      23.7 MB, too large to store) and the seed of
                      tests/conftest.py::pretrained_like_state_dict().
  gdb13_pretrained_like.npz
                      reference loss, APD argmax of every row, a seeded sample of logit entries
                      and per-tensor gradient max/rms/sum for the 256 rows through
                      pretrained_like_state_dict().
  gdb13_pretrained_logits.npz
                      the same for the shipped checkpoint itself (full logits; written by an
                      earlier version of this script, kept as a record).
  live_reference.npz  reference logits of each model on molecules the small fixtures do not
                      hold, and the reference's behaviour on a batch with a multi-type bond.
"""
import hashlib
import json
import os
import sys
from collections import OrderedDict

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from graphinvent_b200 import synthetic as S          # noqa: E402
from oracle import mpnn_oracle as O                  # noqa: E402  (make_constants / kl_loss only)
from tests import refimpl                            # noqa: E402

SMALL = dict(n_node_features=6, n_edge_features=3, max_n_nodes=7, len_f_add_per_node=9,
             len_f_conn_per_node=3, hidden_node_features=12, message_size=10, message_passes=3,
             enn_hidden_dim=20, enn_depth=2, msg_hidden_dim=20, msg_depth=2, att_hidden_dim=18,
             att_depth=2, gather_width=11, gather_att_hidden_dim=16, gather_att_depth=2,
             gather_emb_hidden_dim=14, gather_emb_depth=2, mlp1_hidden_dim=24, mlp1_depth=2,
             mlp2_hidden_dim=28, mlp2_depth=2, edge_emb_size=12, edge_emb_hidden_dim=20,
             edge_emb_depth=2)


def small_constants(model):
    kw = dict(SMALL)
    if model == "MNN":
        kw["message_size"] = 12
    return O.make_constants(model, **kw)


def constants_json(C):
    return json.dumps({k: getattr(C, k) for k in C._fields})


def run_reference(net, nodes, edges, target):
    out = net(nodes, edges)
    loss = O.kl_loss(out, target)          # restated Workflow.py:833-860 (Workflow is not importable)
    net.zero_grad()
    loss.backward()
    grads = OrderedDict((k, p.grad.detach().clone()) for k, p in net.named_parameters())
    return out.detach(), loss.detach(), grads


def make_small(model, seed):
    torch.manual_seed(seed)
    C = small_constants(model)
    net = refimpl.build(C)
    n1, e1 = S.random_graphs(27, C.max_n_nodes, 4, 2, seed=seed + 10, min_atoms=0)
    n2, e2 = S.corner_case_graphs(C.max_n_nodes, C.n_node_features)
    nodes, edges = np.concatenate([n2, n1]), np.concatenate([e2, e1])
    apd = C.max_n_nodes * (C.len_f_add_per_node + C.len_f_conn_per_node) + 1
    target = S.random_targets(nodes.shape[0], apd, seed=seed)
    out, loss, grads = run_reference(net, torch.from_numpy(nodes).float(),
                                     torch.from_numpy(edges).float(), torch.from_numpy(target))
    blob = {"constants": np.array(constants_json(C)), "nodes": nodes, "edges": edges,
            "target": target, "logits": out.numpy(), "loss": loss.numpy()}
    for k, v in net.state_dict().items():
        blob["param/" + k] = v.numpy()
    for k, v in grads.items():
        blob["grad/" + k] = v.numpy()
    np.savez_compressed(os.path.join(HERE, f"small_{model}.npz"), **blob)
    print(model, "rows", nodes.shape[0], "loss", float(loss))


GDB13_SAMPLE = 8192         # logit entries stored out of 256 x 625
STATS_SEED = 20240601


def make_checkpoint_stats():
    path = os.path.join(refimpl.DATA, "fine-tuning", "gdb13_1K-debug", "pretrained_model.pth")
    sd = torch.load(path, map_location="cpu", weights_only=False)
    shapes = np.zeros((len(sd), 2), np.int64)
    for i, v in enumerate(sd.values()):
        shapes[i, :v.dim()] = v.shape
    np.savez_compressed(os.path.join(HERE, "checkpoint_stats.npz"), names=np.array(list(sd)),
                        ndim=np.array([v.dim() for v in sd.values()], np.int64), shapes=shapes,
                        mean=np.array([v.double().mean().item() for v in sd.values()]),
                        std=np.array([v.double().std(unbiased=False).item() for v in sd.values()]),
                        seed=np.int64(STATS_SEED), sha256=np.array(hashlib.sha256(open(path, "rb").read()).hexdigest()))
    print("checkpoint stats:", len(sd), "tensors,", sum(v.numel() for v in sd.values()), "parameters")


def make_gdb13():
    from tests.conftest import pretrained_like_state_dict
    h5 = os.path.join(refimpl.DATA, "pre-training", "gdb13_1K", "train.h5")
    nodes, edges, apds = refimpl.read_gdb13_h5(h5)
    nodes, edges, apds = nodes[:256].copy(), edges[:256].copy(), apds[:256].copy()
    rows = os.path.join(HERE, "gdb13_rows.npz")
    if not os.path.exists(rows):
        np.savez_compressed(rows, nodes=nodes, edges=edges, apds=apds)
    # the file cut to 16 rows: header, then the first 16 rows of the APD / edge / node datasets
    raw = np.fromfile(h5, np.int8)
    n_all = (raw.size - 2048) // (625 + 13 * 13 * 3 + 13 * 8)
    parts, o = [raw[:2048]], 2048
    for row in (625, 13 * 13 * 3, 13 * 8):
        parts.append(raw[o:o + 16 * row])
        o += n_all * row
    np.concatenate(parts).tofile(os.path.join(HERE, "gdb13_train_excerpt.h5"))
    C = O.make_constants("GGNN")
    net = refimpl.build(C)
    net.load_state_dict(pretrained_like_state_dict())
    out, loss, grads = run_reference(net, torch.from_numpy(nodes).float(),
                                     torch.from_numpy(edges).float(),
                                     torch.from_numpy(apds).float())
    idx = np.sort(np.random.default_rng(STATS_SEED).choice(out.numel(), GDB13_SAMPLE, replace=False))
    blob = {"logit_index": idx, "logit_sample": out.numpy().reshape(-1)[idx], "loss": loss.numpy(),
            "argmax": out.argmax(1).numpy().astype(np.int16),
            "grad_names": np.array(list(grads.keys())),
            "grad_absmax": np.array([float(g.abs().max()) for g in grads.values()], np.float32),
            "grad_rms": np.array([float(g.pow(2).mean().sqrt()) for g in grads.values()], np.float32),
            "grad_sum": np.array([float(g.double().sum()) for g in grads.values()], np.float64)}
    # full gradients of a few small / sensitive tensors
    for k in ("gru.bias_ih", "gru.bias_hh", "msg_nns.2.seq.12.bias", "APDReadout.fTermNet2.seq.12.weight",
              "gather.att_nn.seq.0.bias", "msg_nns.0.seq.0.bias"):
        blob["grad/" + k] = grads[k].numpy()
    np.savez_compressed(os.path.join(HERE, "gdb13_pretrained_like.npz"), **blob)
    print("gdb13 x checkpoint-shaped weights: loss", float(loss))


def make_live():
    """per model: reference logits with the small fixture's weights on 24 fresh random molecules; on the multi-type
    bond batch: the error the reference raises (AttentionGGNN, EMN) or its logits (GGNN, default dims, oracle
    seed-2 weights)"""
    from tests.conftest import load_small
    from tests.test_oracle import _multitype_batch
    blob = {}
    for model in ("GGNN", "MNN", "AttGGNN", "EMN"):
        fx = load_small(model)
        C = fx["C"]
        net = refimpl.build(C)
        net.load_state_dict(fx["sd"])
        n, e = S.random_graphs(24, C.max_n_nodes, 4, 2, seed=77, min_atoms=0)
        with torch.no_grad():
            blob[f"logits/{model}"] = net(torch.from_numpy(n).float(), torch.from_numpy(e).float()).numpy()
        Cd = O.make_constants(model)
        net = refimpl.build(Cd)
        net.load_state_dict(O.init_state_dict(Cd, seed=2))
        nodes, edges = _multitype_batch(Cd)
        try:
            with torch.no_grad():
                blob[f"multitype_logits/{model}"] = net(nodes, edges).numpy()
        except Exception as ex:                                   # recorded, not raised
            blob[f"multitype_error/{model}"] = np.array(f"{type(ex).__name__}: {ex}")
    np.savez_compressed(os.path.join(HERE, "live_reference.npz"), **blob)
    print("live reference:", sorted(blob))


if __name__ == "__main__":
    assert refimpl.available(), "set GRAPHINVENT_REFERENCE to a GraphINVENT checkout"
    torch.set_num_threads(8)
    parts = sys.argv[1:] or ["small", "gdb13", "live"]
    if "small" in parts:
        for i, m in enumerate(("GGNN", "MNN", "AttGGNN", "EMN")):
            make_small(m, 100 + i)
    if "gdb13" in parts:
        make_checkpoint_stats()
        make_gdb13()
    if "live" in parts:
        make_live()
