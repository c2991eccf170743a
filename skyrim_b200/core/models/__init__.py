"""Model registry (reference: skyrim/core/models/__init__.py:9-17).  The B200 engine builds the
two step operators the north star names plus GraphCast (BASELINE config 4); the other reference wrappers
(fourcastnet, dlwp, fuxi, fengwu) are not part of this path."""
from .base import GlobalModel, GlobalPrediction, GlobalPredictionRollout  # noqa: F401
from .fourcastnet import FourcastnetModel  # noqa: F401  (not in MODELS yet: the facade's model list is pinned)
from .fourcastnet_v2 import FourcastnetV2Model
from .graphcast import GraphcastModel
from .pangu import PanguModel

MODELS = {"pangu": PanguModel, "fourcastnet_v2": FourcastnetV2Model, "graphcast": GraphcastModel}
