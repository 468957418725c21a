"""B200-native (sm_100a) implementation of the TomoSAR2Height dual-topology hot path.

Public API mirrors the reference package ``tomosar2height`` (model.py, encoder/, decoder/,
block/): ``TomoSAR2Height(cfg)``, ``encoder_dict``, ``decoder_dict``, ``ResnetBlockFC``.
The compute goes through hand-written CUDA kernels in ``csrc/`` behind the C ABI in
``include/t2h.h``; there is no CPU fallback.
"""
from .model import TomoSAR2Height  # noqa: F401
from .decoder import decoder_dict  # noqa: F401
from .encoder import encoder_dict  # noqa: F401
from .block import ResnetBlockFC  # noqa: F401
from .config import berlin_config, munich_config, Config, to_config  # noqa: F401
from .topology import RaggedCloud  # noqa: F401
from .adapters import load_config, ChunkCloud, write_raster, read_raster  # noqa: F401
from .trainer import Trainer  # noqa: F401
from .generator import SceneGenerator, OrthoImage  # noqa: F401
from .evaluation import residual_stats  # noqa: F401


def install_as_reference():
    """Alias this package as ``tomosar2height`` so the reference's train.py / test.py /
    generator.py (``from tomosar2height import TomoSAR2Height``) pick up the B200 path."""
    import sys
    me = sys.modules[__name__]
    sys.modules["tomosar2height"] = me
    for sub in ("model", "encoder", "decoder", "block", "encoder.pointnet", "encoder.alto", "encoder.unet",
                "decoder.pixel", "block.resnet"):
        sys.modules["tomosar2height." + sub] = sys.modules[__name__ + "." + sub]
    return me
