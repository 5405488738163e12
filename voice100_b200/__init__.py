"""voice100_b200: Voice100's batched-inference hot path on hand-written sm_100a CUDA kernels.

Drop-in module names follow the reference (kaiidams/voice100):
    voice100.data_modules.MelSpectrogramAudioTransform -> voice100_b200.MelSpectrogramAudioTransform
    voice100.models.asr.AudioToTextCTC                 -> voice100_b200.AudioToTextCTC
    voice100.models.tts.TextToAlignTextModel           -> voice100_b200.TextToAlignTextModel
    voice100.models.tts.AlignTextToAudioModel          -> voice100_b200.AlignTextToAudioModel
All compute goes through libv100.so (include/v100.h); importing this package does not need a GPU, but
every forward does, and fails loudly otherwise.
"""
from ._lib import V100Error, LIB_PATH  # noqa: F401
from .data_modules import MelSpectrogramAudioTransform, BLANK_AUDIO, LOG_OFFSET, MELSPEC_DIM  # noqa: F401
from .asr import AudioToTextCTC, ConvVoiceEncoder, LinearCharDecoder, AsrPipeline  # noqa: F401
from .tts import (TextToAlignTextModel, AlignTextToAudioModel, VoiceDecoder, WORLDNorm, align_batch,  # noqa: F401
                  TtsPipeline)
from .text import BasicTokenizer, CharTokenizer  # noqa: F401
from .checkpoint import load_checkpoint  # noqa: F401
from .align import ctc_best_path_batch  # noqa: F401
from .kernels import align_frames  # noqa: F401
from .audio import maskaudio  # noqa: F401
from .v2 import (AudioToAlignText, TextToAlignText, AlignTextToAudio, AsrV2Pipeline,  # noqa: F401
                 ConvLayerBlock, ConvTransposeLayerBlock, get_conv_layers, align_batch_v2, TtsV2Pipeline)
from .vocoder import AlignTextToAudioPredict, create_mc2sp_matrix  # noqa: F401
