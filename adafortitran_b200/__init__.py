"""adafortitran_b200 -- B200-native (sm_100a) inference forward pass of AdaFortiTran / FortiTran.

Public surface (mirrors the reference's ``src.models`` / ``src.config``):
    FortiTranEstimator, AdaFortiTranEstimator, BaseFortiTranEstimator, LinearEstimator
    data.extract_values, data.extract_pilots, data.MatDataset, data.collate_on_device   (input side, row N2)
    data.SyntheticChannels                                                             (data generated on the GPU)
    SystemConfig, ModelConfig, load_config
"""
from .config import ConfigLoader, ModelConfig, OFDMParams, PilotParams, SystemConfig, load_config
from .estimators import AdaFortiTranEstimator, BaseFortiTranEstimator, FortiTranEstimator, LinearEstimator

__all__ = [
    "AdaFortiTranEstimator", "BaseFortiTranEstimator", "FortiTranEstimator", "LinearEstimator",
    "SystemConfig", "ModelConfig", "OFDMParams", "PilotParams", "ConfigLoader", "load_config",
]
__version__ = "0.1.0"
