"""edm_tts_b200: B200-native S2A masked iterative decoding + DAC RVQ search behind the reference's Python API.

(The directory is named edm_tts_b200 because "edm-tts_b200" is not an importable Python identifier.)
"""
from .config import DACConfig, InjectionConformerConfig, TextToSemanticWLenConfig  # noqa: F401


def __getattr__(name):
    # torch / CUDA are only touched when the model classes are actually requested
    if name == "InjectionConformerModel":
        from .s2a import InjectionConformerModel
        return InjectionConformerModel
    if name == "TextToSemanticWLen":
        from .t2s import TextToSemanticWLen
        return TextToSemanticWLen
    if name == "ResidualVectorQuantize":
        from .dac_rvq import ResidualVectorQuantize
        return ResidualVectorQuantize
    if name == "DAC":
        from .dac import DAC
        return DAC
    if name == "DACEncoder":
        from .dac_encoder import DACEncoder
        return DACEncoder
    if name in ("HubertFeatures", "SemanticTokenizer"):
        from . import hubert
        return getattr(hubert, name)
    raise AttributeError(name)
