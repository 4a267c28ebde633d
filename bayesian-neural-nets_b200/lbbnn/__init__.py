"""lbbnn -- B200-native (sm_100a) implementation of the variational-layer hot path of
LarsELund/Bayesian-Neural-Nets.  Python host code over the C-ABI of liblbbnn.so (include/lbbnn.h).
CUDA only: importing this package without the built library raises."""
from . import _capi
from ._capi import LbbnnError, philox_normal, philox_uniform
from .lrt import BayesianLinear, BayesianNetwork, LayerConfig, lrt_linear, manual_seed, predict_ensemble
from . import flows, mf, mnf
from .engine import GraphedTrainer, LRTReplicaTrainer, LRTTrainer, LRTTensorCoreTrainer, MultiTensorAdam
from . import vd
from . import predict
from .predict import EnsemblePredictor, mf_outofsample

__all__ = ["BayesianLinear", "BayesianNetwork", "GraphedTrainer", "LayerConfig", "LRTReplicaTrainer", "LRTTrainer", "LRTTensorCoreTrainer", "LbbnnError", "MultiTensorAdam", "lrt_linear",
           "manual_seed", "predict_ensemble", "predict", "EnsemblePredictor", "mf_outofsample", "mf", "mnf", "flows", "vd", "philox_normal", "philox_uniform"]
