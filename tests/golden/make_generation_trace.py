"""
Records a golden trace of the reference's batched graph generator (`GraphGenerator.build_graphs`,
reference GraphGenerator.py:99-161) for the §8(f) generation-round kernels:

    GRAPHINVENT_REFERENCE=<GraphINVENT checkout> python tests/golden/make_generation_trace.py

The unmodified reference `GraphGenerator` is imported with three stub modules (rdkit, MolecularGraph,
parameters.constants -- SURVEY.md Appendix C); the model is the reference GGNN with the shipped checkpoint on CPU.
`torch.distributions.Multinomial.sample` is wrapped to record the one-hot draws, so the trace holds, per round, the
sampled flat APD index and the likelihood the generator stores for it (`apds[one_hot == 1]`) for every slot, plus the generator's final output buffers.  Replaying
the recorded draws through `graphinvent_b200.generation` must reproduce those buffers bit-exactly.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import mpnn_oracle as O     # noqa: E402
from tests import refimpl               # noqa: E402


def install_stubs(C):
    for name in ("rdkit", "rdkit.Chem"):
        sys.modules.setdefault(name, types.ModuleType(name))
    mg = types.ModuleType("MolecularGraph")
    mg.GenerationGraph = type("GenerationGraph", (), {"__init__": lambda self, **kw: None})
    sys.modules["MolecularGraph"] = mg
    pkg = types.ModuleType("parameters")
    pkg.__path__ = []
    pc = types.ModuleType("parameters.constants")
    pc.constants = C
    pkg.constants = pc
    sys.modules["parameters"] = pkg
    sys.modules["parameters.constants"] = pc


def generator_constants(**kw):
    base = O.make_constants("GGNN")._asdict()
    N, A, CH, E = 13, 5, 3, 3
    base.update(dim_nodes=[N, A + CH], dim_edges=[N, N, E], dim_f_add=[N, A, CH, E], dim_f_conn=[N, E],
                n_atom_types=A, n_formal_charge=CH, n_imp_H=0, n_chirality=0, use_explicit_H=False, ignore_H=True,
                use_chirality=False, atom_types=["C", "N", "O", "S", "Cl"], formal_charge=[-1, 0, 1],
                imp_H=[0, 1, 2, 3], chirality=["None", "R", "S"], generation_epoch=1, job_dir="/tmp/")
    base.update(kw)
    from collections import namedtuple
    return namedtuple("constants", sorted(base))(**base)


def main(batch=96, seed=7):
    assert refimpl.available()
    C = generator_constants()
    install_stubs(C)
    refimpl.load()
    import GraphGenerator as GG     # the unmodified reference module
    torch.manual_seed(seed)
    net = refimpl.build(O.make_constants("GGNN"))
    net.load_state_dict(torch.load(os.path.join(refimpl.DATA, "fine-tuning", "gdb13_1K-debug", "pretrained_model.pth"), map_location="cpu",
                                   weights_only=False))
    net.eval()
    draws, liks = [], []
    orig_sample = torch.distributions.Multinomial.sample

    def recording_sample(self, sample_shape=torch.Size()):
        one_hot = orig_sample(self, sample_shape)
        draws.append(one_hot.argmax(1).to(torch.int32).numpy().copy())
        return one_hot

    orig_get_actions = GG.GraphGenerator.get_actions

    def recording_get_actions(self, apds):
        res = orig_get_actions(self, apds)
        liks.append(res[4].numpy().copy())       # `apds[apd_one_hot == 1]`: the values the generator stores
        return res

    GG.GraphGenerator.get_actions = recording_get_actions

    torch.distributions.Multinomial.sample = recording_sample
    try:
        with torch.no_grad():
            gen = GG.GraphGenerator(model=net, batch_size=batch)
            n_generated = gen.build_graphs()
    finally:
        torch.distributions.Multinomial.sample = orig_sample
        GG.GraphGenerator.get_actions = orig_get_actions
    out = dict(batch=np.int32(batch), n_generated=np.int32(n_generated), rounds=np.int32(len(draws)),
               actions=np.stack(draws), likelihoods=np.stack(liks),
               generated_nodes=gen.generated_nodes.numpy().astype(np.int8),
               generated_edges=gen.generated_edges.numpy().astype(np.int8),
               generated_n_nodes=gen.generated_n_nodes.numpy(),
               generated_likelihoods=gen.generated_likelihoods.numpy(),
               properly_terminated=gen.properly_terminated.numpy(),
               final_nodes=gen.nodes.numpy().astype(np.int8), final_edges=gen.edges.numpy().astype(np.int8),
               final_n_nodes=gen.n_nodes.numpy(), final_likelihoods=gen.likelihoods.numpy())
    np.savez_compressed(os.path.join(HERE, "generation_trace.npz"), **out)
    nn = gen.generated_n_nodes[:n_generated].float()
    print(f"rounds {len(draws)}, generated {n_generated}, properly terminated "
          f"{int(gen.properly_terminated[:n_generated].sum())}, mean atoms {nn.mean():.2f}, max {int(nn.max())}")


if __name__ == "__main__":
    main()
