"""Drop-in boundary: register the B200 classes under the reference's registry names.

The reference builds everything through `utils/registry_class.py` singletons
(`MODEL.build(cfg.UNet)`, `DIFFUSION.build(cfg.Diffusion)`, `AUTO_ENCODER.build(cfg.auto_encoder)`,
utils/registry.py:24-72,106-122).  Re-registering an existing name only warns and replaces
(:116-119), so importing this module AFTER `from tools import *` (inference.py:14) swaps the hot path:

    # two lines added to the reference's inference.py (see INTEGRATION.md)
    import vgen_b200
    vgen_b200.register()

When the reference is not importable (tests, bench), `register()` falls back to the minimal mirror
below, which implements the same `build` contract: `cls(**{k: v for k != 'type'}, **kwargs)`.
"""
from __future__ import annotations

import logging
import warnings


class Registry:
    """Mirror of the reference Registry's public behaviour (utils/registry.py:75-155)."""

    def __init__(self, name):
        self.name = name
        self.class_map = {}

    def get(self, req_type):
        return self.class_map.get(req_type)

    def build(self, cfg, **kwargs):
        if not isinstance(cfg, dict):
            raise TypeError(f"config must be type dict, got {type(cfg)}")
        if "type" not in cfg:
            raise KeyError(f"config must contain key type, got {cfg}")
        cfg = dict(cfg)
        req_type = cfg.pop("type")
        cls = self.get(req_type)
        if cls is None:
            raise KeyError(f"{req_type} not found in {self.name} registry")
        try:
            return cls(**cfg, **kwargs)
        except Exception as e:  # same re-raise convention as utils/registry.py:61-65
            raise Exception(f"Failed to init class {cls}, with {e}") from e

    def register_class(self, name=None):
        def _register(cls):
            key = name or cls.__name__
            if key in self.class_map:
                warnings.warn(f"Class {key} already registered by {self.class_map[key]}, will be replaced by {cls}")
            self.class_map[key] = cls
            return cls
        return _register


MODEL = DIFFUSION = AUTO_ENCODER = EMBEDDER = None
USING_REFERENCE_REGISTRY = False


def register(force_local: bool = False):
    """Register the UNets (T2VBase, I2VGen, VideoLCM, TFT2V, SR600, HiGen), DiffusionDDIM(SR), AutoencoderKL and the three
    FrozenOpenCLIP*Embedder classes under the reference's registry names.  Returns (MODEL, DIFFUSION, AUTO_ENCODER); the
    embedder registry is `vgen_b200.registry.EMBEDDER`."""
    global MODEL, DIFFUSION, AUTO_ENCODER, EMBEDDER, USING_REFERENCE_REGISTRY
    from .autoencoder import AutoencoderKL
    from .clip import FrozenOpenCLIPEmbedder, FrozenOpenCLIPTextVisualEmbedder, FrozenOpenCLIPVisualEmbedder
    from .diffusion import DiffusionDDIM
    from .diffusion_gauss import DiffusionDDIMSR
    from .unet import UNetSD_HiGen, UNetSD_I2VGen, UNetSD_SR600, UNetSD_T2VBase, UNetSD_TFT2V, UNetSD_VideoLCM

    regs = None
    emb = None
    if not force_local:
        try:
            from utils.registry_class import AUTO_ENCODER as A, DIFFUSION as D, MODEL as M  # the reference's singletons
            regs = (M, D, A)
            USING_REFERENCE_REGISTRY = True
        except ImportError:  # the reference is not on sys.path: use the local mirror (tests, bench)
            regs = None
        if regs is not None:
            try:
                from utils.registry_class import EMBEDDER as emb  # noqa: N811
            except ImportError:   # an older reference tree without the embedder registry: keep the three above
                emb = None
    if regs is None:
        regs = (MODEL or Registry("MODEL"), DIFFUSION or Registry("DIFFUSION"), AUTO_ENCODER or Registry("AUTO_ENCODER"))
        USING_REFERENCE_REGISTRY = False
    MODEL, DIFFUSION, AUTO_ENCODER = regs
    logging.getLogger("vgen_b200").info("vgen_b200.register: using %s registries",
                                        "the reference's (utils.registry_class)" if USING_REFERENCE_REGISTRY else "local mirror")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # replacing the reference classes is the point
        for cls in (UNetSD_T2VBase, UNetSD_I2VGen, UNetSD_VideoLCM, UNetSD_TFT2V, UNetSD_SR600, UNetSD_HiGen):
            MODEL.register_class()(cls)
        DIFFUSION.register_class()(DiffusionDDIM)
        DIFFUSION.register_class()(DiffusionDDIMSR)
        AUTO_ENCODER.register_class()(AutoencoderKL)
        EMBEDDER = emb if emb is not None else (EMBEDDER or Registry("EMBEDDER"))   # also reachable as vgen_b200.registry.EMBEDDER
        for cls in (FrozenOpenCLIPEmbedder, FrozenOpenCLIPVisualEmbedder, FrozenOpenCLIPTextVisualEmbedder):
            EMBEDDER.register_class()(cls)
    return MODEL, DIFFUSION, AUTO_ENCODER
