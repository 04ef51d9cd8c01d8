"""pytorch_models_b200: B200-native (sm_100a) implementation of the encoder-block hot path of
gau-nernst/pytorch-models — ``transformer.py`` (LayerNorm, MHA, MLP) plus the ViT patch embedding — behind the
reference's module API. Kernels live in ``csrc/`` and are reached through the C-ABI in ``include/b200enc.h``."""
from . import _lib, ops, plans
from .audio2text import Whisper, WhisperDecoder, WhisperEncoder, WhisperPreprocessor
from .image import ViT
from .text import BERT, GPT, GPT2
from .graphs import GraphedStep
from .transformer import MHA, MLP, Decoder, DecoderLayer, Encoder, EncoderLayer, KVCache, invalidate_packed

__all__ = ["MHA", "MLP", "Encoder", "EncoderLayer", "Decoder", "DecoderLayer", "ViT", "WhisperEncoder", "WhisperDecoder",
           "Whisper", "WhisperPreprocessor", "BERT", "GPT", "GPT2", "ops", "plans", "invalidate_packed", "_lib",
           "KVCache", "GraphedStep"]
