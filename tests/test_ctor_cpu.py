"""Constructor / seed / state_dict parity (SURVEY.md §8 a2, a8, b): under the same torch.manual_seed the drop-in classes
must yield the reference's initial network -- same state_dict keys in the same order and bit-identical parameter values --
because the reference seeds each of its 10 networks with torch.manual_seed(i) (LRT:356, MNF:414, MF:518).
tests/golden/ctor.npz holds the keys and fingerprints of the REFERENCE constructors (tests/golden/make_golden.py ctor).
Runs on CPU: constructing the modules launches no kernel."""
import math
import os

import numpy as np
import pytest
import torch

import cases as C

G = np.load(os.path.join(C.GOLDEN, "ctor.npz"))

# The stored "sum" / "abs" fingerprints are torch's fp64 reductions on the machine that wrote ctor.npz, whose summation
# order follows its thread count and vector width; every one lies within 2 u sum|x| (u = 2^-53) of the exactly rounded
# sum.  Here the sums are exactly rounded (math.fsum: the same value on every machine) and must match within SUM_TOL
# sum|x|; shape, head and sample are compared bit for bit.
SUM_TOL = 4 * 2.0 ** -53


def _digest(v):
    f = v.detach().reshape(-1)
    x = f.double().tolist()
    return {"shape": np.array(v.shape, dtype=np.int64), "sum": math.fsum(x), "abs": math.fsum(map(abs, x)),
            "head": f[:8].numpy().copy(), "sample": f[::max(1, f.numel() // 64)].numpy().copy()}


def _assert_matches(v, key, what):
    d = _digest(v)
    for n, val in d.items():
        ref = G[f"{key}|{n}"]
        if n in ("sum", "abs"):
            assert abs(val - float(ref)) <= SUM_TOL * d["abs"], what + (n,)
        else:
            assert np.array_equal(np.asarray(val), ref), what + (n,)


def _check(tag, module, extra=None):
    sd = module.state_dict()
    assert list(sd.keys()) == list(G[tag + "_keys"]), tag
    for k, v in sd.items():
        _assert_matches(v, f"{tag}|{k}", (tag, k))
    for name, layers in (extra or {}).items():
        for li, lay in enumerate(layers):
            _assert_matches(getattr(lay, name), f"{tag}|extra.l{li + 1}.{name}", (tag, name, li))


@pytest.mark.parametrize("seed", [0, 7])
def test_lrt_mnf_mf_networks_initialise_like_the_reference(seed):
    import lbbnn
    torch.manual_seed(seed)
    _check(f"lrt{seed}", lbbnn.BayesianNetwork())
    torch.manual_seed(seed)
    _check(f"mnf{seed}", lbbnn.mnf.BayesianNetwork())
    torch.manual_seed(seed)
    net = lbbnn.mf.BayesianNetwork()
    _check(f"mf{seed}", net, {"gammas": net.layers, "alpha": net.layers})


def test_sim_study_and_iaf_constructors_initialise_like_the_reference():
    import lbbnn
    torch.manual_seed(3)
    net = lbbnn.mf.SimStudyNetwork()
    _check("mfsim3", net, {"gammas": net.layers, "alpha": net.layers})
    torch.manual_seed(3)   # MNFsim:146-184: lambdal ~ U(1.5, 2.5), flows_simstudy hidden sizes [50]*5

    class _Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l1 = lbbnn.mnf.BayesianLinear(20, 1, 2, mu_prior=0.1, sigma_prior=1.3, alpha_prior=0.3, bias_sigma_prior=1.3,
                                               lambda_init=(1.5, 2.5), h_sizes=(50,) * 5)
    _check("mnfsim3", _Net())
    torch.manual_seed(5)
    _check("mnfiaf5", lbbnn.mnf.BayesianLinear(40, 12, 2, z_flow_type="MNF", r_flow_type="MNF"))
