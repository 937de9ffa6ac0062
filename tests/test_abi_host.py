"""CPU: the C-ABI library loads and exports every symbol include/gib200.h declares; host-side
plan / layout logic (pure C++ host code, callable without a GPU); module protocol on CPU."""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

from tests.conftest import MODELS, ROOT, load_small, pretrained_like_state_dict


def test_header_symbols_are_exported_and_bound():
    from graphinvent_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "gib200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(gib_[a-z0-9_]+)\s*\(", hdr)))
    assert declared, "no declarations parsed"
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), f"{name} declared in gib200.h but not exported by libgib200.so"
    assert declared == _lib.exported_symbols()
    assert _lib.lib.gib_version() == _lib.ABI_VERSION
    assert ctypes.sizeof(_lib.Dims) == 27 * 4      # 25 ints + big + in_dtype


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("big", [False, True])
def test_plan_matches_reference_parameter_schema(model, big):
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200._lib import lib
    from graphinvent_b200.gnn import mpnn
    from oracle import mpnn_oracle as O
    kw = dict(hidden_node_features=128, message_size=128, message_passes=4, edge_emb_size=128,
              max_n_nodes=38, n_node_features=12, len_f_add_per_node=81) if big else {}
    C = O.make_constants(model, **kw)
    net = mpnn.create(C)
    shapes = O.param_shapes(C)
    sd = net.state_dict()
    assert [k for k, _ in shapes] == list(sd.keys())
    assert all(tuple(sd[k].shape) == tuple(s) for k, s in shapes)
    d = Fn.make_dims(net, 64)
    assert lib.gib_model_num_params(ctypes.byref(d)) == len(shapes)
    for i, (k, s) in enumerate(shapes):
        assert lib.gib_model_param_numel(ctypes.byref(d), i) == math.prod(s), k
    assert lib.gib_model_packed_bytes(ctypes.byref(d)) >= 4 * sum(math.prod(s) for _, s in shapes)


def test_workspace_queries_scale_with_the_graph_header():
    from graphinvent_b200 import functional as Fn
    from graphinvent_b200._lib import lib
    from graphinvent_b200.gnn import mpnn
    from oracle import mpnn_oracle as O
    net = mpnn.create(O.make_constants("GGNN"))
    d = Fn.make_dims(net, 256)

    def hdr(counts):
        h = np.zeros(16, np.int32)
        base = 0
        for t, c in enumerate(counts):
            h[2 + t], h[6 + t] = c, base
            base += (c + 127) // 128 * 128
        h[6 + len(counts)] = base
        h[0], h[1] = sum(counts), base
        return h

    small, large = hdr([1000, 100, 10]), hdr([4000, 400, 40])
    ws = [lib.gib_model_workspace_bytes(ctypes.byref(d), h.ctypes.data_as(ctypes.c_void_p)) for h in (small, large)]
    assert 0 < ws[0] < ws[1]
    bad = hdr([10, 0, 0]); bad[1] = 0          # P < E: inconsistent header -> refused, not UB
    assert lib.gib_model_workspace_bytes(ctypes.byref(d), bad.ctypes.data_as(ctypes.c_void_p)) == 0
    assert b"inconsistent" in lib.gib_last_error()


def test_modules_refuse_cpu_tensors_and_submodule_calls():
    from graphinvent_b200.gnn import modules, mpnn
    fx = load_small("GGNN")
    net = mpnn.create(fx["C"])
    net.load_state_dict(fx["sd"])                      # golden (reference-initialised) weights load by name
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net(fx["nodes"], fx["edges"])
    with pytest.raises(NotImplementedError):
        net.gather(torch.zeros(1, 7, 12), torch.zeros(1, 7, 6), torch.ones(1, 7))
    with pytest.raises(NotImplementedError):
        modules.MLP(4, [8], 2, 0.0)(torch.zeros(3, 4))


def test_reference_checkpoint_loads_by_name():
    """the shipped checkpoint's tensor names, order and shapes (tests/golden/checkpoint_stats.npz)"""
    from graphinvent_b200.gnn import mpnn
    from oracle import mpnn_oracle as O
    sd = pretrained_like_state_dict()
    net = mpnn.create(O.make_constants("GGNN"))
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    assert sum(p.numel() for p in net.parameters()) == 5914773


def test_dropout_in_training_mode_is_refused():
    from graphinvent_b200.gnn import mpnn
    from oracle import mpnn_oracle as O
    net = mpnn.create(O.make_constants("GGNN", enn_dropout_p=0.1))
    with pytest.raises(NotImplementedError, match="dropout"):
        net(torch.zeros(1, 13, 8), torch.zeros(1, 13, 13, 3))


def test_dropin_install_resolves_gnn_mpnn():
    import sys
    from graphinvent_b200 import dropin
    saved = {k: sys.modules.get(k) for k in ("gnn", "gnn.mpnn", "gnn.modules")}
    try:
        dropin.install()
        import gnn.mpnn as m
        from graphinvent_b200.gnn import mpnn
        assert m.GGNN is mpnn.GGNN and m.AttentionGGNN is mpnn.AttentionGGNN and m.EMN is mpnn.EMN
    finally:
        dropin.uninstall()
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
            else:
                sys.modules.pop(k, None)


def test_synthetic_generator_matches_survey_statistics():
    from graphinvent_b200 import synthetic as S
    for n, want in ((13, 28), (38, 86), (40, 90)):
        nodes, edges = S.random_graphs(200, n, 5, 3, seed=n)
        per = edges.sum() / 200
        assert abs(per - want) <= 2.5, (n, per)
        assert (edges == edges.transpose(0, 2, 1, 3)).all()            # symmetric
        assert edges.sum(-1).max() == 1                                # one-hot bond type
        assert (edges.sum((2, 3)).max(1) <= 4).all()                   # valence
        assert (nodes.sum(-1) == 2).all()                              # atom type + neutral charge
    t = S.random_targets(8, 625, seed=0)
    assert np.allclose(t.sum(1), 1, atol=1e-5) and (t > 0).all()


def test_raw_hdf5_reader_matches_the_golden_rows():
    """gdb13_1K/train.h5 of the reference, cut to its header and first 16 rows (tests/golden/make_golden.py)"""
    import os
    from graphinvent_b200 import data
    path = os.path.join(ROOT, "tests", "golden", "gdb13_train_excerpt.h5")
    assert open(path, "rb").read(8) == b"\x89HDF\r\n\x1a\n"
    nodes, edges, apds = data.read_hdf5_raw(path, 13, 8, 3, 625)
    z = np.load(os.path.join(ROOT, "tests", "golden", "gdb13_rows.npz"))
    assert nodes.shape == (16, 13, 8) and edges.shape == (16, 13, 13, 3) and apds.shape == (16, 625)
    assert (nodes == z["nodes"][:16]).all() and (edges == z["edges"][:16]).all() and (apds == z["apds"][:16]).all()
    with pytest.raises(ValueError):
        data.read_hdf5_raw(path, 13, 8, 3, 624)
