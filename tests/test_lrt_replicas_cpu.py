"""LRTReplicaTrainer and the replica launch's C-ABI (lbbnn_lrt_step_replicas_*) without a GPU: every rejection is raised
before any device call, and the planner's host code gives the replica launch the single network's plan at R = 1."""
import ctypes

import pytest
import torch

import lbbnn
from lbbnn import _capi as K

MNIST = (784, 400, 600, 10)


def _nets(n, sizes=(20, 16, 3), **kw):
    return [lbbnn.BayesianNetwork(sizes, **kw) for _ in range(n)]


@pytest.mark.parametrize("make, match", [
    (lambda: ([torch.nn.Linear(3, 3)], {}), "is not an LRT BayesianNetwork"),
    (lambda: ([], {}), "1..64 networks"),
    (lambda: (_nets(65, (4, 3)), {}), "1..64 networks"),
    (lambda: (_nets(1) + _nets(1, (20, 17, 3)), {}), "has sizes"),
    (lambda: (_nets(1) + _nets(1, alpha_prior=0.25), {}), "priors or var_mode"),
    (lambda: (_nets(1) + _nets(1, var_mode="exact"), {}), "priors or var_mode"),
    (lambda: (_nets(2), dict(batch_size=129)), "batch 1..128"),
    (lambda: (_nets(2), dict(batch_size=0)), "batch 1..128"),
    (lambda: (_nets(2, (8,) * 9 + (3,)), {}), "<= 8 layers"),
    (lambda: (_nets(2), dict(seeds=[1])), "need 2 seeds"),
    (lambda: (_nets(2), dict(seeds=[1, -1])), "need 2 seeds"),
    (lambda: (_nets(2), dict(seeds=[1, 2 ** 64])), "need 2 seeds"),
    (lambda: (_nets(2), {}), "one CUDA device"),
], ids=["not-lrt", "zero-nets", "65-nets", "sizes", "priors", "var-mode", "batch-129", "batch-0", "nine-layers",
        "seed-count", "negative-seed", "seed-past-64-bits", "cpu-nets"])
def test_trainer_rejects_before_any_device_call(make, match, monkeypatch):
    """Each bad argument raises LbbnnError naming it; none of them reaches CUDA (the checks run before require_device)."""
    monkeypatch.setattr(K, "require_device", lambda: pytest.fail("reached the device before rejecting"))
    nets, kw = make()
    kw = dict(dict(batch_size=7, num_batches=600), **kw)
    with pytest.raises(lbbnn.LbbnnError, match=match):
        lbbnn.LRTReplicaTrainer(nets, **kw)


def _step(sizes, batch):
    """An lbbnn_step of the stack with LRTTrainer's flat layout; returns it and one replica's float count."""
    st = K.Step()
    st.n_layers, st.batch = len(sizes) - 1, batch
    off = 0
    for i, (k, n) in enumerate(zip(sizes[:-1], sizes[1:])):
        sl = st.layer[i]
        sl.in_features, sl.out_features = k, n
        nk, n4 = (k * n + 3) // 4 * 4, (n + 3) // 4 * 4
        sl.off_weight_mu, sl.off_weight_rho, sl.off_lambdal = off, off + nk, off + 2 * nk
        sl.off_bias_mu, sl.off_bias_rho = off + 3 * nk, off + 3 * nk + n4
        off += 3 * nk + 2 * n4
        sl.priors, sl.var_mode = K.Priors(0, 1, 0.05, 0, 1), 0
    return st, off


def _replicas(R, stride, **kw):
    rp = K.StepReplicas()
    rp.replicas, rp.param_stride = R, stride
    rp.x_stride, rp.y_stride = kw.get("x_stride", 0), kw.get("y_stride", 0)
    return rp


def _describe(st, rp):
    buf = ctypes.create_string_buffer(4096)
    if K.lib.lbbnn_lrt_step_replicas_describe(st, rp, buf, 4096) != 0:
        raise K.LbbnnError(K.lib.lbbnn_last_error().decode())
    return buf.value.decode()


def _clear_env(monkeypatch):
    for k in ("LBBNN_STEP_GENERIC_HEAD", "LBBNN_STEP_OVERLAP_UPDATE") + tuple(f"LBBNN_STEP_PLAN_L{l}" for l in range(8)):
        monkeypatch.delenv(k, raising=False)


@pytest.mark.parametrize("R, stride_delta, kw, match", [
    (0, 0, {}, "replicas must be 1..64"),
    (65, 0, {}, "replicas must be 1..64"),
    (2, 2, {}, "param_stride must be a positive multiple of 4"),
    (2, -4, {}, "past param_stride"),
    (2, 0, dict(x_stride=-1), "x_stride and y_stride must be >= 0"),
    (2, 0, dict(y_stride=-1), "x_stride and y_stride must be >= 0"),
])
def test_c_abi_rejects_bad_replica_arguments(R, stride_delta, kw, match, monkeypatch):
    _clear_env(monkeypatch)
    st, P = _step(MNIST, 100)
    rp = _replicas(R, P + stride_delta, **kw)
    assert K.lib.lbbnn_lrt_step_replicas_workspace_bytes(st, rp) == 0
    assert match in K.lib.lbbnn_last_error().decode()
    with pytest.raises(K.LbbnnError, match=match):
        _describe(st, rp)
    # and the launch itself, before it touches a device
    assert K.lib.lbbnn_lrt_step_replicas_f32(st, rp, None, 0, None) != 0
    assert match in K.lib.lbbnn_last_error().decode()


def test_c_abi_rejects_a_data_parallel_descriptor(monkeypatch):
    _clear_env(monkeypatch)
    st, P = _step(MNIST, 100)
    dp = K.StepDp()
    dp.world = 2
    st.dp = ctypes.pointer(dp)
    assert K.lib.lbbnn_lrt_step_replicas_workspace_bytes(st, _replicas(2, P)) == 0
    assert "dp must be NULL" in K.lib.lbbnn_last_error().decode()


def test_one_replica_gets_the_single_network_plan_and_workspace(monkeypatch):
    """R = 1 prints exactly lbbnn_lrt_step_describe's schedule and needs the same workspace, also under a forced plan and
    the tiled head; R > 1 appends its replica count and needs more workspace (one block per replica)."""
    for env in ({}, {"LBBNN_STEP_PLAN_L0": "8,5,0,0,0,0"}, {"LBBNN_STEP_GENERIC_HEAD": "1"}):
        _clear_env(monkeypatch)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        st, P = _step(MNIST, 100)
        buf = ctypes.create_string_buffer(4096)
        assert K.lib.lbbnn_lrt_step_describe(st, buf, 4096) == 0
        single = buf.value.decode()
        assert _describe(st, _replicas(1, P)) == single
        assert K.lib.lbbnn_lrt_step_replicas_workspace_bytes(st, _replicas(1, P)) == K.lib.lbbnn_lrt_step_workspace_bytes(st)
        four = _describe(st, _replicas(4, P))
        assert four.endswith(" replicas=4"), four
        assert K.lib.lbbnn_lrt_step_replicas_workspace_bytes(st, _replicas(4, P)) > K.lib.lbbnn_lrt_step_workspace_bytes(st)


def test_many_replicas_choose_the_tiled_head(monkeypatch):
    """The small head keeps at most 8 rows per CTA: at R x B = 3200 rows (> 8 per CTA of 296) the planner picks the tiled
    head, whose loss phase walks any number of rows."""
    _clear_env(monkeypatch)
    st, P = _step(MNIST, 100)
    assert "head=small" in _describe(st, _replicas(10, P))
    assert "head=tiled" in _describe(st, _replicas(32, P))
