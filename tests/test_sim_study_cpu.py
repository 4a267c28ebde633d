"""Argument checks of the one-launch simulation-study trainer that need no GPU: lbbnn.mf.SimStudyEnsemble and the C entry
points reject bad input with LbbnnError before any device call."""
import ctypes

import pytest
import torch

import cases as C  # noqa: F401  (sets sys.path)


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def _nets(lb, R=2, in_features=20):
    return [lb.mf.SimStudyNetwork(in_features=in_features) for _ in range(R)]


def test_cpu_networks_and_data_are_rejected(lb):
    with pytest.raises(lb.LbbnnError, match="CUDA"):
        lb.mf.SimStudyEnsemble(_nets(lb), torch.zeros(800, 20), torch.zeros(800), batch_size=400)


@pytest.mark.parametrize("case", ["rows", "in", "shape", "flags", "X", "y", "lrs", "empty"])
def test_bad_arguments_are_rejected(lb, case):
    nets, X, y, B, kw = _nets(lb), torch.zeros(800, 20), torch.zeros(800), 400, {}
    if case == "rows":
        B = 300
    elif case == "in":
        nets, X = _nets(lb, in_features=40), torch.zeros(800, 40)
    elif case == "shape":
        nets[1] = lb.mf.SimStudyNetwork(in_features=10)
    elif case == "flags":
        nets[1].l1.weight_prior.exact = True
    elif case == "X":
        X = torch.zeros(3, 800, 20)
    elif case == "y":
        y = torch.zeros(801)
    elif case == "lrs":
        kw = {"lrs": {"weight_sigma": 1e-3}}
    elif case == "empty":
        nets = []
    with pytest.raises(lb.LbbnnError):
        lb.mf.SimStudyEnsemble(nets, X, y, batch_size=B, **kw)


def test_c_entry_points_reject_bad_descriptors(lb):
    K = lb._capi
    d = K.MfSim()
    assert K.lib.lbbnn_mfsim_train_f32(ctypes.byref(d), 1, None) != 0
    d.replicas, d.in_features, d.rows, d.batch = 2, 33, 800, 400
    assert K.lib.lbbnn_mfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"in_features" in K.lib.lbbnn_last_error()
    d.in_features, d.batch = 20, 300
    assert K.lib.lbbnn_mfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"multiple" in K.lib.lbbnn_last_error()
    assert K.lib.lbbnn_mfsim_train_f32(ctypes.byref(d), 0, None) != 0
    assert K.lib.lbbnn_philox_std_gamma(-1.0, 10, 0, 0, None, None) != 0
    assert K.lib.lbbnn_philox_std_gamma(1.0, 10, 0, 0, None, None) != 0
