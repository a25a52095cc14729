"""B200-native Bi-Mamba hot path (drop-in for the `mamba_ssm.Mamba` the reference's Phase-6
backend uses).  Import name: this directory is `robust-audio-deepfake-evolution_b200`; because of
the hyphens import it with `importlib.import_module("robust-audio-deepfake-evolution_b200")` or
through the top-level alias module `bimamba_b200`."""
from . import _lib
from .amp import DeviceGradScaler, FusedEMA
from .dist import FlatGradBucket, shard_batch
from .encoder import BiMambaBackend, PN_BiMambas_Encoder, backend_head
from .fusion import DualStreamFusion, SELayer
from .graph import GraphedForward, GraphedTrainStep
from .mamba_simple import Mamba
from .optim import FusedAdamW
from .training import FGM, LoRALinear, Phase6TrainStep, apply_lora, freeze_batch_norm_stats, mixup_batch, mixup_loss
from .ops import (BiMambaInnerFn, CausalConv1dFn, SelectiveScanFn, bimamba_inner_fn, causal_conv1d_fn,
                  selective_scan_fn)

__all__ = [
    "Mamba", "PN_BiMambas_Encoder", "BiMambaBackend", "backend_head", "BiMambaInnerFn", "CausalConv1dFn", "SelectiveScanFn",
    "bimamba_inner_fn", "causal_conv1d_fn", "selective_scan_fn", "install_mamba_ssm_shim",
    "DualStreamFusion", "SELayer", "FGM", "LoRALinear", "Phase6TrainStep", "apply_lora", "freeze_batch_norm_stats", "mixup_batch", "mixup_loss",
    "FlatGradBucket", "shard_batch", "GraphedForward", "GraphedTrainStep", "FusedAdamW",
    "DeviceGradScaler", "FusedEMA",
]


def install_mamba_ssm_shim():
    """Make `from mamba_ssm.modules.mamba_simple import Mamba` (src/models/DualStreamSEMamba.py:43)
    resolve to this package's Mamba, so the reference model code runs unchanged."""
    import sys
    import types

    from . import mamba_simple as ms
    from . import ops

    pkg = types.ModuleType("mamba_ssm")
    mods = types.ModuleType("mamba_ssm.modules")
    opsm = types.ModuleType("mamba_ssm.ops")
    ssi = types.ModuleType("mamba_ssm.ops.selective_scan_interface")
    ssi.selective_scan_fn = ops.selective_scan_fn
    pkg.Mamba = ms.Mamba
    pkg.modules, pkg.ops = mods, opsm
    mods.mamba_simple = ms
    opsm.selective_scan_interface = ssi
    sys.modules.setdefault("mamba_ssm", pkg)
    sys.modules.setdefault("mamba_ssm.modules", mods)
    sys.modules.setdefault("mamba_ssm.modules.mamba_simple", ms)
    sys.modules.setdefault("mamba_ssm.ops", opsm)
    sys.modules.setdefault("mamba_ssm.ops.selective_scan_interface", ssi)
    return pkg
