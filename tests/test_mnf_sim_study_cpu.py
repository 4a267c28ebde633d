"""Checks of the MNF simulation study that need no GPU: lbbnn.mnf.SimStudyNetwork initialises like the reference's sim-study
layer, and lbbnn.mnf.SimStudyEnsemble and the C entry point reject bad input with LbbnnError before any device call."""
import ctypes

import pytest
import torch

import cases as C  # noqa: F401  (sets sys.path)
from test_ctor_cpu import _check


@pytest.fixture(scope="module")
def lb():
    import lbbnn
    return lbbnn


def test_sim_study_network_initialises_like_the_reference(lb):
    torch.manual_seed(3)
    net = lb.mnf.SimStudyNetwork()
    _check("mnfsim3", net)
    assert net.num_batches == 5.0 and "num_batches" not in net.state_dict()


def _nets(lb, R=2, **kw):
    return [lb.mnf.SimStudyNetwork(**kw) for _ in range(R)]


CASES = ["priors", "shape", "transforms", "hidden", "iaf", "in", "T", "width", "var_mode", "num_batches", "X", "y", "rows",
         "lrs_key", "lrs_missing", "lrs_type", "empty"]


@pytest.mark.parametrize("case", CASES)
def test_bad_arguments_are_rejected(lb, case):
    nets, X, y, B, kw = _nets(lb), torch.zeros(800, 20), torch.zeros(800), 400, {}
    if case == "priors":
        nets[1] = lb.mnf.SimStudyNetwork(alpha_prior=0.2)
    elif case == "shape":
        nets[1] = lb.mnf.SimStudyNetwork(in_features=10)
    elif case == "transforms":
        nets[1] = lb.mnf.SimStudyNetwork(num_transforms=3)
    elif case == "hidden":
        nets[1] = lb.mnf.SimStudyNetwork(h_sizes=(50,) * 4)
    elif case == "iaf":
        nets = _nets(lb, z_flow_type="MNF", r_flow_type="MNF")
    elif case == "in":
        nets, X = _nets(lb, in_features=40, h_sizes=(8,)), torch.zeros(800, 40)
    elif case == "T":
        nets = _nets(lb, num_transforms=5, h_sizes=(8,))
    elif case == "width":
        nets = _nets(lb, h_sizes=(65, 8))
    elif case == "var_mode":
        for n in nets:
            n.l1.cfg = lb.lrt.LayerConfig(0.1, 1.3, 0.3, 0.0, 1.3, var_mode="exact")
    elif case == "num_batches":
        nets[1].num_batches = 4.0
    elif case == "X":
        X = torch.zeros(3, 800, 20)
    elif case == "y":
        y = torch.zeros(801)
    elif case == "rows":
        B = 300
    elif case == "lrs_key":
        kw = {"lrs": {**{g: 1e-3 for g in lb.mnf.SIM_GROUPS}, "weight_sigma": 1e-3}}
    elif case == "lrs_missing":
        kw = {"lrs": {"weight_mu": 1e-3}}
    elif case == "lrs_type":
        kw = {"lrs": "1e-3"}
    elif case == "empty":
        nets = []
    with pytest.raises(lb.LbbnnError):
        lb.mnf.SimStudyEnsemble(nets, X, y, batch_size=B, **kw)


def test_cpu_networks_and_data_are_rejected(lb):
    with pytest.raises(lb.LbbnnError, match="CUDA"):
        lb.mnf.SimStudyEnsemble(_nets(lb), torch.zeros(800, 20), torch.zeros(800), batch_size=400)


def test_run_arguments_are_checked_before_any_device_call(lb):
    """epochs, lrs and noise of run() on an ensemble built without a device: each is rejected before the launch."""
    ens = object.__new__(lb.mnf.SimStudyEnsemble)
    ens.R, ens.in_features, ens.n_transforms, ens.rows, ens.batch, ens.lrs = 2, 20, 2, 800, 400, [1e-3] * 12
    ens.flat = torch.zeros(2, 4)
    for bad in (0, -1, 1.5, True):
        with pytest.raises(lb.LbbnnError, match="epochs"):
            ens.run(bad)
    with pytest.raises(lb.LbbnnError, match="lrs"):
        ens.run(1, lrs={"z_flow": 1e-3})
    good = {"eps_z": (2, 2, 20), "eps_z2": (2, 2, 20), "z_masks": (2, 2, 2, 20), "z_masks2": (2, 2, 2, 20),
            "r_masks": (2, 2, 2, 20), "eps": (2, 2, 400), "eps_r": (2, 2)}
    with pytest.raises(lb.LbbnnError, match="exactly"):
        ens.run(1, noise={k: torch.zeros(s) for k, s in good.items() if k != "eps_r"})
    for name in good:
        shapes = dict(good, **{name: good[name][:-1] + (good[name][-1] + 1,)})
        with pytest.raises(lb.LbbnnError, match=name):
            ens.run(1, noise={k: torch.zeros(s) for k, s in shapes.items()})
    with pytest.raises(lb.LbbnnError, match="live on"):          # CPU noise
        ens.run(1, noise={k: torch.zeros(s) for k, s in good.items()})
    assert ens.lrs == [1e-3] * 12                                # a rejected run changes nothing


def test_c_entry_point_rejects_bad_descriptors(lb):
    K = lb._capi
    d = K.MnfSim()
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 1, None) != 0
    d.replicas, d.in_features, d.rows, d.batch, d.n_transforms, d.n_hidden = 2, 33, 800, 400, 2, 5
    for i in range(5):
        d.hidden[i] = 50
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"in_features" in K.lib.lbbnn_last_error()
    d.in_features, d.n_transforms = 20, 5
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"n_transforms" in K.lib.lbbnn_last_error()
    d.n_transforms, d.hidden[2] = 2, 65
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"hidden width" in K.lib.lbbnn_last_error()
    d.hidden[2], d.batch = 50, 300
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 1, None) != 0
    assert b"multiple" in K.lib.lbbnn_last_error()
    assert K.lib.lbbnn_mnfsim_train_f32(ctypes.byref(d), 0, None) != 0
    hid = (ctypes.c_int * 5)(*([50] * 5))
    net = lb.mnf.SimStudyNetwork()
    assert K.lib.lbbnn_mnfsim_param_count(20, 2, 5, hid) == sum(p.numel() for p in net.parameters())
    assert K.MNFSIM_MAX_IN == 32 and K.MNFSIM_MAX_T == 4 and K.MNFSIM_MAX_H == 64
