"""B200-native (sm_100a) waveform generation for Megatts2_HierSpeechpp.

Drop-in replacements for the reference's hot-path modules — the HierSpeech++
BigVGAN-style ``Generator`` + ``SourceNetwork`` and the ``SpeechSR`` 24k/48k
upsamplers — backed by hand-written CUDA kernels behind a C-ABI
(``include/hsv.h`` / ``libhsv.so``).  See DESIGN.md and INTEGRATION.md.
"""
from .modules import (AMPBlock0, AMPBlock1, Activation1d, DBlock, DownSample1d, Generator, LowPassFilter1d,
                      SnakeBeta, SourceNetwork, SpeechSR24, SpeechSR24Generator, SpeechSR48, SpeechSR48Generator,
                      SpeechSRGenerator, UpSample1d, Vocoder, VocoderSR, get_padding, invalidate_caches, kaiser_sinc_filter1d)
from .config import HIER_CFG, SR_CFG
from .runtime import CudaGraphRunner, patch_reference, shard_utterances, to_pcm16
from .sr_stream import SpeechSRStream
from .resample import Resample, SpeechSRAudio
from . import front, ops, ttv
from .front import HierSpeechSynthesizer
from .ttv import PitchPredictor, TTVTail, W2VDecoder

__all__ = [
    "AMPBlock0", "AMPBlock1", "Activation1d", "DBlock", "DownSample1d", "Generator", "LowPassFilter1d", "SnakeBeta",
    "SourceNetwork", "SpeechSR24", "SpeechSR24Generator", "SpeechSR48", "SpeechSR48Generator", "SpeechSRGenerator",
    "UpSample1d", "Vocoder", "VocoderSR", "get_padding", "kaiser_sinc_filter1d", "HIER_CFG", "SR_CFG", "CudaGraphRunner",
    "patch_reference", "shard_utterances", "ops", "front", "HierSpeechSynthesizer", "invalidate_caches", "to_pcm16",
    "ttv", "W2VDecoder", "PitchPredictor", "TTVTail", "SpeechSRStream",
    "Resample", "SpeechSRAudio",
]
