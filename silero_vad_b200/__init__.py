"""silero_vad_b200 -- B200-native (sm_100a) Silero-VAD inference engine with the reference's Python surface.

    from silero_vad_b200 import load_silero_vad, get_speech_timestamps, VADIterator
    model = load_silero_vad()
    segments = get_speech_timestamps(wav, model)

(The directory is `silero_vad_b200` because a hyphen cannot appear in a Python package name.)
"""
__version__ = "0.1.0"

from .model import SileroVADB200, load_silero_vad
from .tuning import (VADDecoderRNNJIT, calculate_best_thresholds, decoder_state_dict, encoder_features, export_weights, predict, save_tuned,
                     train, validate, write_container)
from .utils_vad import (VADIterator, VADIteratorBatch, collect_chunks, collect_chunks_batch, drop_chunks, get_speech_timestamps,
                        get_speech_timestamps_batch, read_audio, save_audio)

__all__ = ["SileroVADB200", "load_silero_vad", "get_speech_timestamps", "get_speech_timestamps_batch", "VADIterator", "VADIteratorBatch",
           "collect_chunks", "collect_chunks_batch", "drop_chunks", "read_audio", "save_audio",
           "VADDecoderRNNJIT", "encoder_features", "decoder_state_dict", "train", "validate", "predict", "calculate_best_thresholds",
           "save_tuned", "export_weights", "write_container"]
