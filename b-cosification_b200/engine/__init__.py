"""Fused execution plans over the C-ABI kernels (CUDA only; no fallback)."""
from .resnet import PRECISION_MODES, PipelinedExplainer, ResNetPlan  # noqa: F401
from .train import DenseNetTrainPlan, ResNetTrainPlan  # noqa: F401
from .clip_rn import CLIPResNetPlan  # noqa: F401
from .clip_train import CLIPResNetTrainPlan  # noqa: F401
from .vit import ViTPlan  # noqa: F401
from .densenet import DenseNetPlan  # noqa: F401
from .clip_vit import CLIPViTPlan  # noqa: F401
