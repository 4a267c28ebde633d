"""Reference of the MNF simulation-study objective, built on the oracle's MNF layer (oracle/lbbnn_oracle.py:
mnf_forward): the float64 truth of tests/test_mnf_sim_study_gpu.py and the float32 host port of
profiles/bench_mnf_sim_study.py.  Test infrastructure only."""
import torch
import torch.nn.functional as F

import cases as C  # noqa: F401  (sets sys.path)
import lbbnn_oracle as O


def mnfsim_loss(x, y, p, noise, num_batches, priors=O.Priors(), kind="RNVP"):
    """lbbnn.mnf.SimStudyNetwork.loss with every draw injected: one in -> 1 MNF layer, sigmoid output, BCELoss(sum),
    loss = nll + kl / num_batches -- the MF study's objective (MFsim:258, 287) with the MNF layer's kl (MNF:263-275).
    y: (B,) {0, 1} targets.  Returns (loss, nll, kl, out)."""
    act, kl = O.mnf_forward(x, p, noise, priors=priors, kind=kind)
    out = torch.sigmoid(act)
    nll = F.binary_cross_entropy(out, y.reshape(out.shape).to(out.dtype), reduction="sum")
    return nll + kl / num_batches, nll, kl, out
