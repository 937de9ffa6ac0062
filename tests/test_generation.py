"""§8(f) rank 1: the device-side generation round against a trace of the unmodified reference generator.
The trace (tests/golden/generation_trace.npz, made by tests/golden/make_generation_trace.py) holds the draws the
reference sampled in every round and its final buffers; replaying the draws must reproduce the buffers bit-exactly."""
import os

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN


def _trace():
    return np.load(os.path.join(GOLDEN, "generation_trace.npz"))


def test_trace_fixture_is_self_consistent():
    z = _trace()
    B, n_gen, R = int(z["batch"]), int(z["n_generated"]), int(z["rounds"])
    assert z["actions"].shape == (R, B) and z["likelihoods"].shape == (R, B)
    assert B <= n_gen <= 2 * B and R < 26
    assert 0 <= z["actions"].min() and z["actions"].max() <= 624
    nn = z["generated_n_nodes"][:n_gen]
    atoms = (z["generated_nodes"][:n_gen].sum(-1) > 0).sum(-1)
    assert (atoms == nn).all()                                   # node rows agree with the atom counts
    assert (z["generated_edges"][:n_gen] == z["generated_edges"][:n_gen].transpose(0, 2, 1, 3)).all()
    assert z["properly_terminated"][:n_gen].sum() >= n_gen // 3  # trained checkpoint: most molecules terminate properly


def test_generation_oracle_replays_the_reference_trace_bit_exactly():
    """pins oracle/generation_oracle.py to the unmodified reference generator (CPU, no GPU needed)"""
    from oracle import generation_oracle as G
    z = _trace()
    B = int(z["batch"])
    st = G.GenerationState(B, 13, 5, 3, 3)
    for rnd, (a, l) in enumerate(zip(z["actions"], z["likelihoods"])):
        G.generation_round(st, rnd, a, l)
    assert st.n_generated == int(z["n_generated"])
    assert (st.generated_nodes.astype(np.int8) == z["generated_nodes"]).all()
    assert (st.generated_edges.astype(np.int8) == z["generated_edges"]).all()
    assert (st.generated_n_nodes == z["generated_n_nodes"]).all()
    assert (st.generated_likelihoods == z["generated_likelihoods"]).all()
    assert (st.properly_terminated == z["properly_terminated"]).all()
    assert (st.nodes.astype(np.int8) == z["final_nodes"]).all() and (st.edges.astype(np.int8) == z["final_edges"]).all()
    assert (st.n_nodes.astype(np.int8) == z["final_n_nodes"]).all() and (st.likelihoods == z["final_likelihoods"]).all()


def _action_stream(rng, st, apd, len_add):
    """per slot, mostly a valid-looking add (bond to an existing atom; overflows once the graph is full) so graphs grow
    to max_n_nodes; the remaining 0.6/N of the draws are connects among existing atoms (valid, self loop or duplicate
    bond), connects to a random position (missing atom), terminates and uniformly random indices"""
    B, N, A, CH, Ef = st.B, st.N, st.A, st.CH, st.Ef
    q = 0.6 / N
    u = rng.random(B)
    n = st.n_nodes
    big = rng.integers(0, 1 << 30, B)
    bond_to = np.where(n > 0, big % np.maximum(n, 1), 0)
    first_bond = np.where((n == 0) & (rng.random(B) < 0.9), 0, rng.integers(0, Ef, B))
    add = ((bond_to * A + rng.integers(0, A, B)) * CH + rng.integers(0, CH, B)) * Ef + np.where(n == 0, first_bond, rng.integers(0, Ef, B))
    conn_in = len_add + bond_to * Ef + rng.integers(0, Ef, B)
    conn_any = len_add + rng.integers(0, N, B) * Ef + rng.integers(0, Ef, B)
    a = np.where(u < 1 - q, add,
                 np.where(u < 1 - 0.5 * q, conn_in,
                          np.where(u < 1 - 0.3 * q, conn_any, np.where(u < 1 - 0.15 * q, apd - 1, rng.integers(0, apd, B)))))
    return a.astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("seed,N,A,CH,Ef,B", [(0, 13, 5, 3, 3, 200), (1, 5, 2, 1, 2, 64), (2, 38, 9, 3, 3, 96)])
def test_round_kernels_match_the_oracle_on_random_action_streams(seed, N, A, CH, Ef, B):
    """a synthetic action stream that grows graphs up to max_n_nodes and hits every validity rule (bond to a missing
    atom, first atom off slot 0, full graph, connect in an empty graph, self loop, double bond) far more often than
    a trained model does"""
    from graphinvent_b200.config import make_constants
    from graphinvent_b200.generation import GraphGenerator
    from oracle import generation_oracle as G
    rng = np.random.default_rng(seed)
    C = make_constants("GGNN", max_n_nodes=N, n_node_features=A + CH, n_edge_features=Ef,
                       len_f_add_per_node=A * CH * Ef, len_f_conn_per_node=Ef)
    apd = N * (A * CH * Ef + Ef) + 1
    rounds = 2 * N - 1
    liks = rng.random((rounds, B)).astype(np.float32)
    st = G.GenerationState(B, N, A, CH, Ef)
    gen = GraphGenerator(model=None, batch_size=B, constants=C, n_atom_types=A, n_formal_charge=CH)
    len_add = N * A * CH * Ef
    for rnd in range(rounds):
        if st.n_generated > B:          # a round writes at most B-1 graphs: stay inside the 2B output buffers
            break
        a = _action_stream(rng, st, apd, len_add)
        G.generation_round(st, rnd, a, liks[rnd])
        # drive the kernels one round at a time through the same entry point build_graphs() uses
        import ctypes
        from graphinvent_b200._lib import check, lib
        P = lambda t: ctypes.c_void_p(t.data_ptr())
        ad, ld = torch.from_numpy(a).cuda(), torch.from_numpy(liks[rnd]).cuda()
        check(lib.gib_generation_round(B, N, A + CH, Ef, A, CH, rnd, P(ad), P(ld), P(gen.nodes), P(gen.edges),
                                       P(gen.n_nodes), P(gen.likelihoods), P(gen.generated_nodes),
                                       P(gen.generated_edges), P(gen.generated_n_nodes), P(gen.generated_likelihoods),
                                       P(gen.properly_terminated), gen.capacity, P(gen._counters), P(gen._scratch),
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "round")
        assert int(gen._counters[0].item()) == st.n_generated, rnd
        assert (gen.nodes.cpu().numpy() == st.nodes).all(), rnd
        assert (gen.edges.cpu().numpy() == st.edges).all(), rnd
        assert (gen.n_nodes.cpu().numpy() == st.n_nodes).all(), rnd
        assert (gen.likelihoods.cpu().numpy() == st.likelihoods).all(), rnd
    assert (gen.generated_nodes.cpu().numpy() == st.generated_nodes).all()
    assert (gen.generated_edges.cpu().numpy() == st.generated_edges).all()
    assert (gen.generated_n_nodes.cpu().numpy() == st.generated_n_nodes).all()
    assert (gen.generated_likelihoods.cpu().numpy() == st.generated_likelihoods).all()
    assert (gen.properly_terminated.cpu().numpy() == st.properly_terminated).all()
    assert st.n_generated > B // 4 and int(st.generated_n_nodes.max()) == N     # the stream filled graphs completely


@pytest.mark.gpu
def test_replay_reproduces_the_reference_generator_bit_exactly():
    from graphinvent_b200.config import make_constants
    from graphinvent_b200.generation import GraphGenerator
    z = _trace()
    B, n_gen = int(z["batch"]), int(z["n_generated"])
    C = make_constants("GGNN")
    gen = GraphGenerator(model=None, batch_size=B, constants=C, n_atom_types=5, n_formal_charge=3)
    replay = [(torch.from_numpy(a), torch.from_numpy(l)) for a, l in zip(z["actions"], z["likelihoods"])]
    got = gen.build_graphs(replay=replay)
    assert got == n_gen and gen.rounds == int(z["rounds"])
    assert torch.equal(gen.generated_nodes.cpu().to(torch.int8), torch.from_numpy(z["generated_nodes"]))
    assert torch.equal(gen.generated_edges.cpu().to(torch.int8), torch.from_numpy(z["generated_edges"]))
    assert torch.equal(gen.generated_n_nodes.cpu(), torch.from_numpy(z["generated_n_nodes"]))
    assert torch.equal(gen.generated_likelihoods.cpu(), torch.from_numpy(z["generated_likelihoods"]))
    assert torch.equal(gen.properly_terminated.cpu(), torch.from_numpy(z["properly_terminated"]))
    # the live batch state after the last round too (incl. the dummy graph's accumulated bonds)
    assert torch.equal(gen.nodes.cpu().to(torch.int8), torch.from_numpy(z["final_nodes"]))
    assert torch.equal(gen.edges.cpu().to(torch.int8), torch.from_numpy(z["final_edges"]))
    assert torch.equal(gen.n_nodes.cpu().to(torch.int8), torch.from_numpy(z["final_n_nodes"]))
    assert torch.equal(gen.likelihoods.cpu(), torch.from_numpy(z["final_likelihoods"]))


@pytest.mark.gpu
def test_attention_ggnn_generation_survives_a_multi_type_bond_in_the_dummy_slot():
    """Slot 0 (the dummy graph) is never reset and accumulates every action it samples: two "add" actions with
    different bond types leave a bond with two non-zero types, on which the reference's AggregationMPNN prologue (and
    this package's AttentionGGNN) raise.  The generator evaluates the dummy graph on a sanitised copy instead of dying
    and keeps the reference's state of slot 0."""
    from graphinvent_b200.config import make_constants
    from graphinvent_b200.generation import GraphGenerator
    from graphinvent_b200.gnn import mpnn
    C = make_constants("AttGGNN")
    torch.manual_seed(3)
    net = mpnn.create(C).cuda().eval()
    gen = GraphGenerator(net, batch_size=64, n_atom_types=5, n_formal_charge=3)
    # the state after the dummy graph sampled add(bond_to=0, single) and add(bond_to=0, double) in two rounds
    gen.nodes[0, 1, 0] = 1.0; gen.nodes[0, 1, 6] = 1.0
    for t in (0, 1):
        gen.edges[0, 0, 1, t] = 1.0; gen.edges[0, 1, 0, t] = 1.0
    with pytest.raises(RuntimeError):               # the raw state is what the module itself rejects
        net(gen.nodes, gen.edges)
    g = torch.Generator(device="cuda").manual_seed(1)
    (nodes, edges, n_nodes), flat, final, proper = gen.sample(generator=g)
    assert nodes.shape[0] == 64 and torch.isfinite(final).all()
    assert ((gen.edges[0] != 0).sum(-1) > 1).any().item()          # slot 0 keeps its (reference) state
