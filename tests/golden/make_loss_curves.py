"""
Golden training curves: the UNMODIFIED reference modules (CPU fp32) trained for 50 steps of
`Workflow.train_epoch` (Workflow.py:785-796: zero_grad -> forward -> KL loss -> backward -> Adam step, then the
OneCycleLR step of Workflow.py:245-261) on the tiny-dims fixture batches of `small_<MODEL>.npz`.

    GRAPHINVENT_REFERENCE=<GraphINVENT checkout> python tests/golden/make_loss_curves.py

Output `loss_curves.npz`: per model the 50 losses and the final logits.  SURVEY.md 8c lists "loss curve over 50 Adam
steps within 1e-4" among the tolerances to hold.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import mpnn_oracle as O                  # noqa: E402  (kl_loss only)
from tests import refimpl                            # noqa: E402
from tests.conftest import MODELS, load_small        # noqa: E402

STEPS, LR, MAX_LR = 50, 1e-4, 1e-3


def main():
    assert refimpl.available()
    out = {"steps": np.int32(STEPS), "lr": np.float32(LR), "max_lr": np.float32(MAX_LR)}
    for model in MODELS:
        fx = load_small(model)
        net = refimpl.build(fx["C"])
        net.load_state_dict(fx["sd"])
        net.train()
        opt = torch.optim.Adam(net.parameters(), lr=LR)
        sch = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=MAX_LR, total_steps=STEPS)
        losses = []
        for _ in range(STEPS):
            net.zero_grad()
            loss = O.kl_loss(net(fx["nodes"], fx["edges"]), fx["target"])
            loss.backward()
            opt.step()
            sch.step()
            losses.append(float(loss))
        with torch.no_grad():
            final = net(fx["nodes"], fx["edges"])
        out[f"loss/{model}"] = np.array(losses, np.float64)
        out[f"final_logits/{model}"] = final.numpy()
        print(model, "loss", losses[0], "->", losses[-1])
    np.savez_compressed(os.path.join(HERE, "loss_curves.npz"), **out)


if __name__ == "__main__":
    main()
