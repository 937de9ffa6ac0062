"""
Records a golden trace of the reference's RL rollout generator (`GraphGeneratorRL.build_graphs`, reference
GraphGeneratorRL.py:109-172) and of the gradient that `Workflow.learning_step` (Workflow.py:569-612) sends back
through the whole rollout:

    GRAPHINVENT_REFERENCE=<GraphINVENT checkout> python tests/golden/make_generation_rl_trace.py

The unmodified reference `GraphGeneratorRL` is imported with the stub modules of `make_generation_trace.py`.
agent = reference GGNN with tests/conftest.py::pretrained_like_state_dict() (train mode, as in learning_step);
prior = the same weights plus a seeded perturbation (so that the two likelihood streams differ).  Weights of that kind
terminate almost every molecule within two rounds, so the draws are not sampled from the agent: the generator is fed
the draws of generation_rl_trace.npz, which were sampled by the shipped trained checkpoint
(data/fine-tuning/gdb13_1K-debug/pretrained_model.pth, 16 rounds); the rollout reproduces that trace's buffers, and
generation_rl_trace_pretrained_like.npz receives what depends on the weights.  Recorded per round: the flat APD
index and the agent / prior likelihoods the generator stores for it; at the end: the generator's buffers, the
log-likelihoods `sample()` returns (:92-97, restated without the RDKit conversion), the loss of
`Workflow.compute_loss_component` (:889-896) on fixed pseudo-scores and, per parameter tensor of both models, the
norm of its gradient (plus the full gradient of every tensor with <= 1024 elements).
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from oracle import mpnn_oracle as O                         # noqa: E402
from tests import refimpl                                   # noqa: E402
from make_generation_trace import generator_constants, install_stubs   # noqa: E402

SIGMA = 20.0
PRIOR_SEED, PRIOR_NOISE = 123, 0.02


def perturbed(sd, seed=PRIOR_SEED, noise=PRIOR_NOISE):
    """the prior's weights: agent's + noise * randn, tensor by tensor in state_dict order (CPU generator)"""
    g = torch.Generator().manual_seed(seed)
    return {k: v + noise * torch.randn(v.shape, generator=g) for k, v in sd.items()}


def pseudo_scores(n):
    return torch.tensor([((i * 37) % 10) / 10.0 for i in range(n)], dtype=torch.float32)


def main(batch=40, seed=11):
    assert refimpl.available()
    C = generator_constants()
    install_stubs(C)
    refimpl.load()
    import GraphGeneratorRL as GG                            # the unmodified reference module
    torch.manual_seed(seed)
    forced = np.load(os.path.join(HERE, "generation_rl_trace.npz"))["actions"]
    from tests.conftest import pretrained_like_state_dict
    sd = pretrained_like_state_dict()
    agent = refimpl.build(O.make_constants("GGNN"))
    agent.load_state_dict(sd)
    prior = copy.deepcopy(agent)
    prior.load_state_dict(perturbed(sd))
    agent.train()
    prior.eval()
    draws, liks_a, liks_p = [], [], []
    orig_sample = torch.distributions.Multinomial.sample

    def recording_sample(self, sample_shape=torch.Size()):
        one_hot = torch.zeros_like(self.probs)
        one_hot[torch.arange(one_hot.shape[0]), torch.from_numpy(forced[len(draws)]).long()] = 1
        draws.append(one_hot.argmax(1).to(torch.int32).numpy().copy())
        return one_hot

    orig_get_actions = GG.GraphGeneratorRL.get_actions

    def recording_get_actions(self, agent_apds, prior_apds):
        res = orig_get_actions(self, agent_apds=agent_apds, prior_apds=prior_apds)
        liks_a.append(res[4].detach().numpy().copy())
        liks_p.append(res[5].detach().numpy().copy())
        return res

    GG.GraphGeneratorRL.get_actions = recording_get_actions
    torch.distributions.Multinomial.sample = recording_sample
    try:
        gen = GG.GraphGeneratorRL(model=agent, batch_size=batch)
        gen.agent_model, gen.prior_model = agent, prior
        n_generated = gen.build_graphs()
    finally:
        torch.distributions.Multinomial.sample = orig_sample
        GG.GraphGeneratorRL.get_actions = orig_get_actions
    # GraphGeneratorRL.sample :92-97
    agent_ll = torch.log(torch.sum(gen.generated_agent_likelihoods, dim=1)[:batch])
    prior_ll = torch.log(torch.sum(gen.generated_prior_likelihoods, dim=1)[:batch])
    # Workflow.compute_loss_component :889-896 (uniqueness = 1) and the mean of generate_graphs_rl :752-756
    scores = pseudo_scores(batch)
    diff = agent_ll - (prior_ll + SIGMA * scores)
    loss = torch.mean(diff * diff)
    loss.backward()
    out = dict(batch=np.int32(batch), n_generated=np.int32(n_generated), rounds=np.int32(len(draws)),
               actions=np.stack(draws), agent_likelihoods=np.stack(liks_a), prior_likelihoods=np.stack(liks_p),
               generated_nodes=gen.generated_nodes.numpy().astype(np.int8),
               generated_edges=gen.generated_edges.numpy().astype(np.int8),
               generated_n_nodes=gen.generated_n_nodes.numpy(),
               generated_agent_likelihoods=gen.generated_agent_likelihoods.detach().numpy(),
               generated_prior_likelihoods=gen.generated_prior_likelihoods.detach().numpy(),
               properly_terminated=gen.properly_terminated.numpy(),
               agent_loglikelihoods=agent_ll.detach().numpy(), prior_loglikelihoods=prior_ll.detach().numpy(),
               loss=np.float32(loss.item()), sigma=np.float32(SIGMA), prior_seed=np.int32(PRIOR_SEED),
               prior_noise=np.float32(PRIOR_NOISE))
    for tag, net in (("agent", agent), ("prior", prior)):
        names, norms = [], []
        for k, p in net.named_parameters():
            names.append(k)
            norms.append(float(p.grad.norm()))
            if p.numel() <= 1024:
                out[f"grad_{tag}/{k}"] = p.grad.numpy().copy()
        out[f"grad_norm_{tag}"] = np.array(norms, np.float64)
        out[f"grad_names_{tag}"] = np.array(names)
    # the draws and buffers are those of generation_rl_trace.npz; store what the weights decide
    keep = {k: v for k, v in out.items()
            if "likelihood" in k or k.startswith("grad_") or k in ("loss", "sigma", "prior_seed", "prior_noise")}
    np.savez_compressed(os.path.join(HERE, "generation_rl_trace_pretrained_like.npz"), **keep)
    nn = gen.generated_n_nodes[:n_generated].float()
    print(f"rounds {len(draws)}, generated {n_generated}, properly terminated "
          f"{int(gen.properly_terminated[:n_generated].sum())}, mean atoms {nn.mean():.2f}, max {int(nn.max())}, "
          f"loss {loss.item():.4f}, |grad agent| {np.linalg.norm(out['grad_norm_agent']):.4f}, "
          f"|grad prior| {np.linalg.norm(out['grad_norm_prior']):.4f}")


if __name__ == "__main__":
    main()
