"""honk2_b200 -- B200-native (sm_100a) implementation of honk2's batched keyword-spotting
inference path: the AudioProcessor MFCC front-end plus the forward pass of model.ResNet /
model.CNN, behind honk2's own class_registry + config-dict construction API.

Importing the package registers ``model.ResNet`` and ``model.CNN`` in this package's registry
(same contract as /root/reference/utils/class_registry.py); ``install_into(register_cls)``
re-registers them into an unmodified honk2 checkout (overwrite semantics, utils/trie.py:21).
"""
from .class_registry import register_cls, find_cls, install_into  # noqa: F401
from .torch_utils import calculate_conv_output_size, calculate_pool_output_size  # noqa: F401
from .audio_processor import AudioProcessor  # noqa: F401
from .model import BaseModel, ResNet, CNN  # noqa: F401
from .zoo import MODEL_ZOO, model_config  # noqa: F401
from ._native import NativeError  # noqa: F401
from .profile import profile_layers  # noqa: F401
from .workspace import load_checkpoint, strip_data_parallel_prefix  # noqa: F401
from .streaming import n_stream_windows, stream_window_targets, evaluate_stream, LiveStreams  # noqa: F401
from .data_loader import AudioDataLoader  # noqa: F401
from . import metric  # noqa: F401  (registers metric.Acc, metric.PerClassAcc, loss_fn.ce_loss)

__version__ = "0.1.0"


def build_model(name, n_labels=None, precision=None, seed=None):
    """Construct a zoo model exactly as run/test.py:60-64 does: find_cls("model.<Name>")(config)
    after torch.manual_seed(seed) (run/run_utils.py:15-18), eval mode."""
    import torch
    kind, cfg = model_config(name, n_labels)
    if precision is not None:
        cfg["precision"] = precision
    torch.manual_seed(MODEL_ZOO[name]["seed"] if seed is None else seed)
    m = find_cls(f"model.{kind}")(cfg)
    m.eval()
    return m
