"""audio-calm_b200: B200-native (sm_100a) log-mel front-end and mel statistics pass for Audio-CALM.

The directory name carries a hyphen (it is mandated by the build contract), so the importable name is
``audio_calm_b200``: the repository root holds a small ``audio_calm_b200.py`` loader that registers this
directory as that package.  Layout:

    csrc/acb_kernels.cu      hand-written CUDA kernels + the extern "C" ABI (include/audiocalm_b200.h)
    csrc/acb_dftgemm.cu      tensor-core route: STFT as a split-fp16 DFT-GEMM on tcgen05 (Whisper-style preset)
    whisper.py               WhisperLogMel: WhisperFeatureExtractor-compatible features on that route
    _lib.py                  nvcc build + ctypes binding (fails loudly when the .so is missing)
    tables.py                window / slaney filterbank, bit-identical to the reference's torch tables
    frontend.py              LogMelFrontend: batched + ragged launches, fused peak-norm / affine / moments
    stats.py                 per-bin moments, single all-reduce, finalise like compute_mel_stats.py
    sharding.py              utterance sharding across ranks (length-balanced)
    collate.py               training-feed collation on the device (crop / zero-pad to 256 frames; ragged pad + transpose)
    spectral.py              VAE-side STFT magnitudes over the mel time axis (AcousticVAE._stft_mag / stft_loss forward)
    csrc/acb_spectral.cu     its kernel (shares the in-register FFT-32 of csrc/acb_fft32.cuh)
    resample.py              Resampler: torchaudio.transforms.Resample (sinc_interp_hann) on the device, uniform and ragged
    csrc/acb_resample.cu     its polyphase kernel (banded per-phase coefficients in registers)
    flac.py                  FlacDecoder: FLAC (RFC 9639) streams decoded bit-exact on the device, many per launch
    csrc/acb_flac.cu         its frame-parallel decoder (sync search + CRC-8, one thread per frame, CRC-16, coverage check)
    preprocess/              drop-in mirrors of the reference's preprocess/{core,compute_mel_stats,process_dataset}.py
"""
from . import _lib, tables  # noqa: F401
from .frontend import (LogMelFrontend, MEL_MEAN_DEFAULT, MEL_STD_DEFAULT, RaggedBatch, empty_ragged,  # noqa: F401
                       frames_for_length, pack_clips, padded_frames)
from .stats import MelStats, MelStatsAccumulator, finalize_moments, normalize_per_utterance  # noqa: F401
from . import collate, frontend, stats, sharding  # noqa: F401
from .collate import crop_collate, pad_collate, pad_collate_packed  # noqa: F401
from . import spectral, whisper  # noqa: F401
from .whisper import WhisperLogMel, whisper_tables  # noqa: F401
from . import resample  # noqa: F401
from .resample import Resampler, resampled_length  # noqa: F401
from . import flac  # noqa: F401
from .flac import FlacDecoder, FlacError, FlacInfo, parse_flac  # noqa: F401

__all__ = ["LogMelFrontend", "MelStatsAccumulator", "MelStats", "RaggedBatch", "pack_clips", "frames_for_length",
           "padded_frames", "finalize_moments", "normalize_per_utterance", "MEL_MEAN_DEFAULT", "MEL_STD_DEFAULT", "WhisperLogMel", "whisper_tables",
           "Resampler", "resampled_length", "empty_ragged", "FlacDecoder", "FlacError", "FlacInfo", "parse_flac"]
__version__ = "0.1.0"
