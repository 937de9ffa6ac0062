"""§8(f) rank 1 (RL twin) + rank 4: the two-model rollout of `GraphGeneratorRL` (reference GraphGeneratorRL.py:109-172)
with autograd through the whole rollout (Workflow.learning_step, Workflow.py:569-612).

Pin: tests/golden/generation_rl_trace.npz, recorded from the unmodified reference by
tests/golden/make_generation_rl_trace.py (agent = conftest.pretrained_like_state_dict(), prior = those weights + seeded
noise, draws of a rollout of the shipped trained checkpoint): draws
and both likelihood streams of every round, final buffers, log-likelihoods, the loss of compute_loss_component and the
gradient norms of both models."""
import copy
import os
import types

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN, pretrained_like_state_dict
from tests.test_generation import _action_stream

N, A, CH, EF = 13, 5, 3, 3


def _trace():
    return np.load(os.path.join(GOLDEN, "generation_rl_trace.npz"))


def _trace_pretrained_like():
    """the trace's draws and buffers with what the reference computed for conftest.pretrained_like_state_dict()"""
    z = dict(_trace())
    z.update(np.load(os.path.join(GOLDEN, "generation_rl_trace_pretrained_like.npz")))
    return z


def test_rl_oracle_replays_the_reference_rl_trace_bit_exactly():
    """pins the two-stream mode of oracle/generation_oracle.py to the unmodified reference `GraphGeneratorRL`"""
    from oracle import generation_oracle as G
    z = _trace()
    B, R = int(z["batch"]), int(z["rounds"])
    assert z["actions"].shape == (R, B) and z["agent_likelihoods"].shape == (R, B) == z["prior_likelihoods"].shape
    st = G.GenerationState(B, N, A, CH, EF, rl=True)
    for r in range(R):
        G.generation_round(st, r, z["actions"][r], z["agent_likelihoods"][r], z["prior_likelihoods"][r])
    assert st.n_generated == int(z["n_generated"]) >= B
    assert (st.generated_nodes.astype(np.int8) == z["generated_nodes"]).all()
    assert (st.generated_edges.astype(np.int8) == z["generated_edges"]).all()
    assert (st.generated_n_nodes == z["generated_n_nodes"]).all()
    assert (st.generated_likelihoods == z["generated_agent_likelihoods"]).all()
    assert (st.generated_prior_likelihoods == z["generated_prior_likelihoods"]).all()
    assert (st.properly_terminated == z["properly_terminated"]).all()
    ll = np.log(st.generated_likelihoods.sum(1)[:B])
    assert np.abs(ll - z["agent_loglikelihoods"]).max() <= 1e-6
    # the fixture's loss really is compute_loss_component on these log-likelihoods (Workflow.py:889-896)
    scores = np.array([((i * 37) % 10) / 10.0 for i in range(B)], np.float32)
    diff = z["agent_loglikelihoods"] - (z["prior_loglikelihoods"] + float(z["sigma"]) * scores)
    assert abs(float(np.mean(diff * diff)) - float(z["loss"])) <= 1e-4 * float(z["loss"])


class _TinyAPD(torch.nn.Module):
    """stand-in model for the host-logic test: any differentiable map (nodes, edges) -> APD logits"""

    def __init__(self, apd, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.w = torch.nn.Parameter(0.3 * torch.randn(N * (A + CH) + N * N * EF, apd, generator=g))
        self.b = torch.nn.Parameter(0.1 * torch.randn(apd, generator=g))
        self.graphs_seen = []

    def dims(self):
        return {"model": "GGNN", "N": N, "F": A + CH, "Ef": EF}

    def forward(self, nodes, edges, graph=None):
        self.graphs_seen.append(graph)
        return torch.cat([nodes.flatten(1), edges.flatten(1)], dim=1) @ self.w + self.b


@pytest.mark.parametrize("seed", [0, 1])
def test_rl_generator_host_logic_on_cpu_shims(monkeypatch, seed):
    """GraphGeneratorRL's own logic (slot-id tags through the round kernel, gather of the differentiable per-round
    likelihoods, padding, replay, shared K0, snapshot of the batch before each forward) with the kernels played by
    the numpy oracle: values and gradients must equal an explicit per-(molecule, round) bookkeeping."""
    from oracle import generation_oracle as G
    from tests import hostshim
    from graphinvent_b200.config import make_constants
    from graphinvent_b200.generation import GraphGeneratorRL
    hostshim.install_generation_shims(monkeypatch)
    B = 24
    C = make_constants("GGNN")
    apd = N * (A * CH * EF + EF) + 1
    agent, prior = _TinyAPD(apd, 10 + seed), _TinyAPD(apd, 20 + seed)
    gen = GraphGeneratorRL(None, B, constants=C, n_atom_types=A, n_formal_charge=CH, device="cpu")
    rng = np.random.default_rng(seed)
    used = []

    def stream():                                        # actions that grow molecules, computed from the live batch
        while True:
            live = types.SimpleNamespace(B=B, N=N, A=A, CH=CH, Ef=EF, n_nodes=gen.n_nodes.numpy().copy())
            a = _action_stream(rng, live, apd, N * A * CH * EF)
            used.append(a)
            yield torch.from_numpy(a)

    (nodes, edges, n_nodes), agent_ll, prior_ll, proper = gen.sample(agent, prior, replay=stream())
    R = gen.rounds
    assert R == len(used) and R >= N                     # molecules were grown to max_n_nodes before the batch filled
    assert all(g is not None for g in agent.graphs_seen) and agent.graphs_seen == prior.graphs_seen   # one K0 per round
    w = torch.linspace(0.5, 1.5, B)
    (agent_ll * w).sum().backward(retain_graph=True)
    (prior_ll * w).sum().backward()

    # ---- explicit bookkeeping: state machine = oracle, likelihood owner = unique (round, slot) ids -------------
    agent2, prior2 = copy.deepcopy(agent), copy.deepcopy(prior)
    agent2.zero_grad()
    prior2.zero_grad()
    st = G.GenerationState(B, N, A, CH, EF, rl=True)
    ids = G.GenerationState(B, N, A, CH, EF)
    la, lp = [], []
    for r in range(R):
        nd, ed = torch.from_numpy(st.nodes.copy()), torch.from_numpy(st.edges.copy())
        idx = torch.from_numpy(used[r]).long().unsqueeze(1)
        la.append(torch.softmax(agent2(nd, ed), 1).gather(1, idx).squeeze(1))
        lp.append(torch.softmax(prior2(nd, ed), 1).gather(1, idx).squeeze(1))
        G.generation_round(st, r, used[r], la[-1].detach().numpy(), lp[-1].detach().numpy())
        G.generation_round(ids, r, used[r], (r * B + np.arange(B) + 1).astype(np.float32))
    assert st.n_generated == int(gen._counters[0]) >= B
    assert (gen.generated_nodes.numpy() == st.generated_nodes).all() and (gen.generated_edges.numpy() == st.generated_edges).all()
    assert (gen.generated_n_nodes.numpy() == st.generated_n_nodes).all()
    assert (gen.properly_terminated.numpy() == st.properly_terminated).all()
    assert np.abs(gen.generated_agent_likelihoods.detach().numpy() - st.generated_likelihoods).max() <= 1e-7
    assert np.abs(gen.generated_prior_likelihoods.detach().numpy() - st.generated_prior_likelihoods).max() <= 1e-7
    assert gen.generated_agent_likelihoods.shape == (2 * B, 2 * N)
    exp_a, exp_p = [], []
    for g in range(B):
        terms_a, terms_p = [], []
        for t in range(2 * N):
            k = int(ids.generated_likelihoods[g, t])
            if k:
                r, b = divmod(k - 1, B)
                assert r == t                                 # likelihoods sit at the global round index
                terms_a.append(la[r][b])
                terms_p.append(lp[r][b])
        exp_a.append(torch.log(torch.stack(terms_a).sum()))
        exp_p.append(torch.log(torch.stack(terms_p).sum()))
    exp_a, exp_p = torch.stack(exp_a), torch.stack(exp_p)
    assert (exp_a - agent_ll).abs().max().item() <= 1e-6 and (exp_p - prior_ll).abs().max().item() <= 1e-6
    (exp_a * w).sum().backward()
    (exp_p * w).sum().backward()
    for m, m2 in ((agent, agent2), (prior, prior2)):
        for p, p2 in zip(m.parameters(), m2.parameters()):
            assert p.grad is not None and p.grad.abs().max().item() > 0
            assert (p.grad - p2.grad).abs().max().item() <= 1e-5 * max(1.0, p2.grad.abs().max().item())
    # without a replay the agent's own samples drive the rollout (sampler shim), and nothing needs grad under no_grad
    with torch.no_grad():
        out = gen.sample(agent, prior, generator=torch.Generator().manual_seed(3))
    assert not out[1].requires_grad and torch.isfinite(out[1]).all() and int(gen._counters[0]) >= B


class _OracleModel(torch.nn.Module):
    """the CPU oracle's functional forward behind the module call protocol (parameters = the state_dict)"""

    def __init__(self, C, sd):
        super().__init__()
        self.C = C
        self.names = list(sd)
        self.params = torch.nn.ParameterList([torch.nn.Parameter(v.clone()) for v in sd.values()])

    def forward(self, nodes, edges, graph=None):
        from oracle import mpnn_oracle as O
        return O.forward(dict(zip(self.names, self.params)), self.C, nodes, edges)


def test_rl_generator_with_oracle_models_reproduces_the_reference_trace(monkeypatch):
    """end to end on CPU: this package's GraphGeneratorRL (round kernel played by the generation oracle, models
    played by the MPNN oracle with the checkpoint-shaped weights) replays the reference's draws and must land on the
    reference's own numbers -- both likelihood streams, the log-likelihoods, the RL loss and the gradients that
    flow back through all 16 rounds into both models"""
    from oracle import mpnn_oracle as O
    from tests import hostshim
    from graphinvent_b200.config import make_constants
    from graphinvent_b200.generation import GraphGeneratorRL
    hostshim.install_generation_shims(monkeypatch)
    z = _trace_pretrained_like()
    B, n_gen, R = int(z["batch"]), int(z["n_generated"]), int(z["rounds"])
    sd = pretrained_like_state_dict()
    g = torch.Generator().manual_seed(int(z["prior_seed"]))
    sd_prior = {k: v + float(z["prior_noise"]) * torch.randn(v.shape, generator=g) for k, v in sd.items()}
    C = O.make_constants("GGNN")
    agent, prior = _OracleModel(C, sd), _OracleModel(C, sd_prior)
    gen = GraphGeneratorRL(None, B, constants=make_constants("GGNN"), n_atom_types=A, n_formal_charge=CH, device="cpu")
    _, agent_ll, prior_ll, proper = gen.sample(agent, prior, replay=[torch.from_numpy(a) for a in z["actions"]])
    assert gen.rounds == R and int(gen._counters[0]) == n_gen
    assert (gen.generated_nodes.numpy().astype(np.int8) == z["generated_nodes"]).all()
    assert (gen.generated_edges.numpy().astype(np.int8) == z["generated_edges"]).all()
    assert (gen.properly_terminated.numpy() == z["properly_terminated"]).all()
    assert np.abs(gen.generated_agent_likelihoods.detach().numpy() - z["generated_agent_likelihoods"]).max() <= 5e-6
    assert np.abs(gen.generated_prior_likelihoods.detach().numpy() - z["generated_prior_likelihoods"]).max() <= 5e-6
    assert np.abs(agent_ll.detach().numpy() - z["agent_loglikelihoods"]).max() <= 1e-5
    assert np.abs(prior_ll.detach().numpy() - z["prior_loglikelihoods"]).max() <= 1e-5
    scores = torch.tensor([((i * 37) % 10) / 10.0 for i in range(B)])
    diff = agent_ll - (prior_ll + float(z["sigma"]) * scores)
    loss = torch.mean(diff * diff)
    assert abs(loss.item() - float(z["loss"])) <= 1e-4 * float(z["loss"])
    loss.backward()
    for tag, net in (("agent", agent), ("prior", prior)):
        ref = dict(zip([str(s) for s in z[f"grad_names_{tag}"]], z[f"grad_norm_{tag}"]))
        total = float(np.linalg.norm(z[f"grad_norm_{tag}"]))
        for k, p in zip(net.names, net.params):
            assert abs(p.grad.norm().item() - ref[k]) <= 1e-3 * ref[k] + 1e-5 * total, (tag, k)
            key = f"grad_{tag}/{k}"
            if key in z:
                want = torch.from_numpy(z[key])
                assert (p.grad - want).norm().item() <= 1e-3 * want.norm().item() + 1e-5 * total, (tag, k)
